// lsmrc_kernels.cuh -- fused uplink-receiver kernels for sm_100a.
//
// One kernel template replaces the reference's whole per-symbol chain of library
// calls and tiny kernels (gpuLS.cu, SURVEY.md 2b).  Two fused modes do the work
// (a third, MODE_FFT, is the stand-alone batched transform behind gpuLS::batchedFFT):
//
//   MODE_PILOT : CP strip -> N-pt FFT -> drop DC -> LS divide by the pilot ->
//                conj -> store Hconj[a][k] and sum_a |H|^2
//                (dropPrefix :143 + cuFFT :377 + findHs :158 + findDistSqrd :185;
//                 CPU: cpuLS.hpp:247-317)
//   MODE_DATA  : CP strip -> N-pt FFT -> drop DC -> x conj(H) -> sum over
//                antennas in registers -> / sum|H|^2 -> ascending-frequency
//                store -> hard QAM demap -> packed bits
//                (cuFFT :441 + multiplyWithChannelConj :212 + combineForMRC :236
//                 + shiftOneRow :109; CPU: cpuLS.hpp:319-389; demap is new)
//
// Decomposition of one N-point row transform (Cooley-Tukey, decimation in
// frequency, N = P * R2 * R3):
//   a "team" of T = N/P threads owns a row; every thread keeps P points in
//   registers.  Stage 1 loads x[n1*T + t] straight from global memory (64-bit
//   coalesced loads that skip the cyclic prefix), runs a P-point register DFT
//   over n1, applies W_N^(t*k1) and writes row k1 of a [P][T+1] shared tile.
//   Stage 2 reads the tile transposed (lanes run over k1, stride T+1 complex:
//   conflict free), runs R2-point DFTs; for three-stage plans the result goes
//   back in place with W_(T)^(m2*k2) applied and stage 3 runs R3-point DFTs.
//   After the last stage lane order equals bin order (bin = c + (N/R_last)*j),
//   so the Hconj reads, the combined-symbol stores and the MRC accumulators
//   are all coalesced / register resident: the antenna reduction never leaves
//   the register file (no shared or global intermediate, unlike
//   gpuLS.cu:212-259 which writes and re-reads the full [S][A][K] tensor).
//
// N = 1024 uses P = 32, R2 = 32: one warp per row, warp-level syncs only.
//
// Data kernel structure (details at the code): persistent CTAs pulling work items
// from a global ticket counter; per item each team loops over the antennas with the
// MRC accumulators in registers; for N = 1024 the teams of a CTA share every Hconj
// row through a shared-memory ring filled by bulk async copies (TMA) on mbarriers;
// inter-stage twiddles are fetched a chunk ahead of their use.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "fft_radix.cuh"

constexpr int kHStages = 3;  // depth of the Hconj ring (rows)
constexpr int kTwChunk = 4;  // inter-stage twiddles fetched this many at a time, one chunk ahead of their use

namespace lsmrc {

enum { MODE_PILOT = 0, MODE_DATA = 1, MODE_FFT = 2, MODE_ONESHOT = 3 };

struct KernelParams {
    // input: antenna-samples, complex64.  element (f, s, a, n) at
    //   rx + f*frame_stride + s*sym_stride + a*ant_stride + n   (n includes the CP)
    const float2* rx;
    // one-launch kernel only, frames read in place from the shared-memory ring: the frames of the launch are
    // consecutive ring slots (slot f*S + s); slots >= split_sym continue at rx2 (the run wraps around the end of
    // the ring).  split_sym = INT_MAX: ordinary addressing through frame_stride.
    const float2* rx2;
    int split_sym;
    int x_tma;      // antenna rows are 16-byte aligned: bulk copies allowed
    int rx_align4;  // one-launch kernel only: samples are only 4-byte aligned (slots behind the ring's 12-byte header)
    long long frame_stride;
    long long sym_stride;
    int ant_stride;
    int cp;
    int first_sym;  // symbol index of work item 0 inside a frame (0 pilot, 1 first data)
    int n_ant;      // A
    int n_sym_work; // symbols handled per frame by this launch (1 for pilot, S-1 for data)
    int n_frames;
    int qam_bits;
    // per-frame channel state.  hwork [F][A][N]: conj of the LS estimate indexed by FFT bin
    // (entry 0 unused), 16-byte aligned rows -- the layout the data kernel streams.  hconj
    // [F][A][K] is the reference's layout (bin k+1 at index k, gpuLS.cu:158-182), written only
    // when the caller asks for it (may be nullptr).  hsqrd [F][K] = sum_a |H|^2.
    float2* hwork;
    float2* hconj;
    float* hsqrd;
    // pilot kernel only: antenna groups per frame, partial-energy scratch [F][G][N], arrival counters [F]
    int n_groups;
    int pilot_grid_cap;  // pilot launch: largest grid (one resident wave); 0 = one CTA per virtual CTA
    int frames_per_cta;  // pilot kernel: frames sharing one CTA (> 1 only with n_groups == 1, few antennas)
    float* epart;
    unsigned int* counters;
    // data kernel only: ticket[0] = work-item counter (a CTA's next item is atomicAdd(&ticket[0], 1)), ticket[1] = CTAs
    // that have drawn their last ticket.  Both are zero between launches: the last CTA to leave resets them, so a
    // launch carries no host-side state (safe to replay from a CUDA graph or to move between streams).
    unsigned long long* ticket;
    // single-launch kernel of the shuffle-stage plans (lsmrc_frames_sh): ready[f] = launch number (ticket[2] + 1) once frame
    // f's channel state is complete
    unsigned int* ready;
    // data kernel, plans without the Hconj ring: antennas of one (frame, symbol) are split over
    // ant_split teams of the CTA (power of two, <= TEAMS) whose partial sums are added in shared
    // memory -- used when there are too few (frame, symbol) pairs to fill the GPU (latency configs)
    int ant_split;
    const float2* pilot_bin;  // X in FFT-bin order, K entries (bin k+1 at index k)
    // outputs of MODE_DATA
    float2* combined;  // [F][n_sym_work][K], ascending frequency
    uint8_t* bits;     // [F][n_sym_work][row_bytes] or nullptr
    int bits_row_bytes;
    // optional soft output: max-log LLRs [F][n_sym_work][K][qam_bits] (ascending frequency, bit order as
    // in the packed bits; LLR > 0 <=> bit 0), scaled by sum|H|^2 / noise_var
    float* llr;
    float inv_noise_var;
    const float2* twiddles;  // plan table: tw1 [(P-1)][T] then tw2 [(R2-1)][R3]
};

template <int N_, int P_, int R2_, int R3_, int TEAMS_, int NBUF_ = 2, int PF_X_ = 0, int PF_H_ = 0, int REG_PF_ = 0, bool H_RING_ = false,
          bool X_TMA_ = false, bool TW_TMEM_ = false, int SH_ = 1>
struct Plan {
    // SH > 1 (2 or 4; N = 32 * 32 * SH, teams of SH warps): the LAST radix-SH stage runs across the SH adjacent lanes
    // of a warp through shuffles instead of a second shared-memory exchange (see row_fft).  Measured on B200
    // (tools/ubench_lsu.cu, profiles/r02_ubench_lsu.txt): a 64-bit LDS/STS costs 2 clocks of the SM's L1/LSU data
    // pipe per warp, a SHFL about 0.55, and that pipe is what bounds these kernels.  Consequences of the layout:
    //  * thread (k1, q), q = lane % SH, ends up with bins k1 + 32*k2 + 1024*k3 for 32/SH values of k2 and all k3
    //    (bin_of below), so the per-antenna channel rows are kept slot-major ([slot][thread], hpos below) to stay
    //    coalesced, and
    //  * some outputs carry a unit factor u in {1, -1, i, -i} that depends on (slot, lane) only (unfix/fix below).
    //    The pilot kernel stores conj(H) computed from the same factored outputs, so u cancels in Y * conj(H);
    //    only exported values (Hconj in the reference layout, the stand-alone FFT) are corrected.
    static constexpr int SH = SH_;
    static_assert(SH_ == 1 || ((SH_ == 2 || SH_ == 4) && P_ == 32 && R2_ == 32 && R3_ == 1), "shuffle stage: N = 32*32*SH");
    // TW_TMEM (data kernel, 32 points per thread, CTAs of four warps): the inter-stage twiddles W_N^(t*k1) of a
    // thread are not re-read from the shared-memory table for every row but kept in the thread's tensor-memory lane
    // (see tmem_load8): 31 fewer 64-bit shared loads per thread and row on the pipe that bounds these kernels.
    static constexpr bool TW_TMEM = TW_TMEM_;
    static_assert(!TW_TMEM_ || (P_ == 32 && (N_ / P_) * TEAMS_ == 128), "TW_TMEM: 32 points per thread, four warps per CTA");
    // X_TMA (teams of whole warps): the data kernel brings each antenna row into the team's tile with one bulk
    // async copy (TMA), issued while the previous row is still in its last-stage arithmetic, instead of 64-bit
    // loads into registers at the top of the row.  The copy lays the row out linearly over the first N
    // elements of the (padded, P x (T+1)) tile; the lanes read their samples from there (conflict-free) and the
    // tile is then reused in place as the exchange buffer.
    static constexpr bool X_TMA = X_TMA_;
    // REG_PF: data kernel loads row a+1 into registers right after stage 1 of row a (0 = off, 1 = on).  Pays for the
    // 16-points-per-thread plans; the 32-point plans would need a 255-register budget.
    static constexpr int REG_PF = REG_PF_;
    // H_RING: the TEAMS teams of a CTA work on TEAMS data symbols of ONE frame and share each
    // Hconj row through a shared-memory ring filled by bulk async copies (TMA) on mbarriers
    static constexpr bool H_RING = H_RING_;
    static constexpr int H_STAGES = kHStages;   // ring depth
    static constexpr int H_AHEAD = kHStages - 2; // rows kept in flight ahead of the row being consumed
    static constexpr int TW_CHUNK = (P_ >= 8) ? kTwChunk : P_;  // inter-stage twiddles fetched this many at a time
    static constexpr int HRING = H_RING_ ? H_STAGES * N_ : 0;  // complex elements
    // PF_X: rows ahead whose antenna-samples are prefetched into L2; PF_H: rows ahead whose
    // Hconj row is prefetched into L1 (0 = off)
    static constexpr int PF_X = PF_X_, PF_H = PF_H_;
    static constexpr int N = N_, P = P_, R2 = R2_, R3 = R3_, TEAMS = TEAMS_, NBUF = NBUF_;
    static constexpr int T = N / P;        // threads per team == M1 (points per row of the tile)
    // Tile row pitch (complex elements).  Plain plans pad the row by one element: their stage-2 read has lanes k1 at
    // k1*ROW + const, conflict-free for odd ROW.  Shuffle-stage plans keep the rows dense (so that a whole antenna
    // row lands in the tile with ONE linear bulk copy) and swizzle the columns instead: element (r, c) sits in column
    // c ^ swz(r), swz(r) = SH * (r mod 16/SH).  Their stage-2 read has lanes (k1, q) on column n2*SH + q of row k1,
    // i.e. on bank pair ((n2 ^ k1) mod 16/SH) * SH + q: distinct over the 16 lanes of a 64-bit wavefront.
    static constexpr int ROW = (SH_ > 1) ? T : T + 1;
    static __host__ __device__ constexpr int swz(int r) { return (SH_ > 1) ? SH_ * (r % (16 / SH_)) : 0; }
    // index of element (r, c) of the tile
    static __device__ __forceinline__ int at(int r, int c) { return r * ROW + (c ^ swz(r)); }
    static_assert(!X_TMA_ || (NBUF_ == 1 && N_ / P_ >= 16), "X_TMA: one tile per team, teams of at least half a warp");
    static_assert(!X_TMA_ || ((P_ * (N_ / P_ + 1)) % 2 == 0), "X_TMA: team tiles must stay 16-byte aligned");
    static_assert(!X_TMA_ || H_RING_, "X_TMA: the data kernel sets up the row barriers with the Hconj ring's");
    static constexpr int NB2 = P / R2;     // stage-2 butterflies per thread
    static constexpr int NB3 = P / R3;     // stage-3 butterflies per thread (R3 > 1)
    static constexpr int RL = (R3 > 1) ? R3 : R2;  // radix of the last shared-memory stage
    static constexpr int NBL = P / RL;             // last-stage butterflies per thread
    static constexpr int THREADS = T * TEAMS;
    static constexpr int TW1 = (P - 1) * T;
    static constexpr int TW2 = (SH_ > 1) ? 32 * SH_ : (R3 > 1) ? (R2 - 1) * R3 : 0;  // SH: W_T^(q*k2) at [k2][q]
    static constexpr int TWN = TW1 + TW2;
    static constexpr int TILE = P * ROW;   // complex elements per tile
    // Per-team tile block.  Teams narrower than a half-warp share 64-bit shared-memory wavefronts
    // (16 lanes each): lanes (team j, t) must fall on distinct bank pairs, i.e. j*TEAM_STRIDE + t must
    // be distinct mod 16, which TEAM_STRIDE = T (mod 16) gives.  (An unpadded block is a multiple
    // of 16 elements for the small plans: every team of a warp on the same banks, 4- to 8-way conflicts.)
    static constexpr int TEAM_TILES = NBUF * TILE;
    static constexpr int TEAM_STRIDE = (T >= 16) ? TEAM_TILES : TEAM_TILES + ((T - TEAM_TILES % 16) + 16) % 16;
    static constexpr size_t SMEM_BYTES = sizeof(float2) * (size_t)(TWN + HRING + TEAMS * TEAM_STRIDE);
    static_assert(!H_RING_ || TWN % 2 == 0, "ring rows must stay 16-byte aligned");
    static_assert(P * R2 * R3 * SH_ == N, "plan must factor N");
    // FFT bin of accumulator slot `sl` of thread `t` of a team (the order the sink of row_fft is called in)
    static __device__ __forceinline__ int bin_of(int sl, int t)
    {
        if constexpr (SH_ == 1) {
            return t + T * (sl / RL) + (N / RL) * (sl % RL);
        } else {
            const int lane = t & 31, q = lane % SH_, k1 = lane / SH_ + (32 / SH_) * (t >> 5);
            const int c = sl & 1, kk = brev<32>(sl & ~1);
            const int k2 = kk + 16 * (SH_ == 2 ? q : (q >> 1));
            const int k3 = SH_ == 2 ? c : (q & 1) + 2 * c;
            return k1 + 32 * k2 + 1024 * k3;
        }
    }
    // position of that bin's conj(H) inside a channel row of hwork (N entries per antenna)
    static __device__ __forceinline__ int hpos(int sl, int t, int bin) { return SH_ == 1 ? bin : sl * T + t; }
    // row_fft hands slot `sl` of thread `t` the value y' = u * Y; unfix() returns Y = conj(u) * y', refix() u * v
    template <bool CONJ>
    static __device__ __forceinline__ float2 unit_mul(int sl, int t, float2 v)
    {
        if constexpr (SH_ == 1) {
            return v;
        } else if constexpr (SH_ == 2) {
            const bool neg = (sl & 1) && (t & 1);
            return neg ? make_float2(-v.x, -v.y) : v;
        } else {
            if (!(t & 1)) return v;
            // u = i * kappa (kappa = +-1): u*v = kappa*(-v.y, v.x), conj(u)*v = kappa*(v.y, -v.x)
            const float kappa = (((t >> 1) & 1) != (sl & 1)) ? -1.f : 1.f;
            return CONJ ? make_float2(kappa * v.y, -kappa * v.x) : make_float2(-kappa * v.y, kappa * v.x);
        }
    }
    static __device__ __forceinline__ float2 unfix(int sl, int t, float2 v) { return unit_mul<true>(sl, t, v); }
    static __device__ __forceinline__ float2 refix(int sl, int t, float2 v) { return unit_mul<false>(sl, t, v); }
    // stage-1 outputs of thread t are written with this sign: it swaps, per reading lane, which register of a
    // pair (2j, 2j+1) the last stage-2 butterfly leaves X[k] and X[k+16] in, so that every lane of a shuffle group
    // keeps register 2j and sends register 2j+1 without a select (the sign of the odd-indexed inputs of a
    // decimation-in-time transform flips the sign of the last stage's twiddles)
    static __device__ __forceinline__ float stage1_sign(int t)
    {
        if constexpr (SH_ == 2) return ((t & 3) == 3) ? -1.f : 1.f;
        else if constexpr (SH_ == 4) return ((t & 6) == 6) ? -1.f : 1.f;
        else return 1.f;
    }
    static_assert(P >= R2 && P >= R3, "thread must own whole butterflies");
    static_assert(THREADS <= 1024, "block too large");
    static_assert(T <= 32 || TEAMS <= 15, "named barriers 1..15");
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// streaming 64-bit load of one antenna-sample: read once, keep it out of L1
__device__ __forceinline__ float2 ld_stream(const float2* p)
{
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}

// shared-memory 64-bit load the compiler may not move or merge (used to pin prefetch distance)
__device__ __forceinline__ float2 lds_volatile(const float2* p)
{
    float2 r;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(smem_u32(p)));
    return r;
}

// software prefetch hints: pull lines that a later iteration will read into L2 / L1 so that
// the demand loads of that iteration see cache latency instead of HBM latency
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// each thread of a team touches every 128-byte line of [base, base + n_elems) once
template <int T, bool TO_L1>
__device__ __forceinline__ void prefetch_row(const float2* base, int n_elems, int t)
{
    constexpr int PER_LINE = 128 / (int)sizeof(float2);
#pragma unroll 4
    for (int e = t * PER_LINE; e < n_elems; e += T * PER_LINE) {
        if (TO_L1) prefetch_l1(base + e);
        else prefetch_l2(base + e);
    }
}

// ---- mbarrier + bulk async copy (TMA, 1-D) primitives ---------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// try_wait may put the warp to sleep until the phase completes.  ptxas hoists the first probe of a wait loop far up
// into the arithmetic ahead of it (seen in SASS: into the middle of the preceding transform), where a sleeping probe
// stalls work that does not depend on the barrier at all -- so the first probe is the non-blocking test_wait, and
// the sleeping form is only used inside the loop, which stays where the program has it.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    if (mbar_test_wait(bar, parity)) return;
    while (!mbar_try_wait(bar, parity)) {
    }
}
// global -> shared bulk copy, completion signalled on `bar` (bytes and addresses multiples of 16)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// L2 eviction priorities for bulk copies.  Antenna samples are read exactly once: evict_first keeps them from pushing
// out the channel rows (hwork), which every data symbol of a frame re-reads and which should be served from L2.
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}

// orders this thread's earlier generic-proxy accesses to shared memory before later async-proxy (bulk copy) ones
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tensor memory as a per-thread constant store --------------------------------------------------------
// The FFT twiddles of a thread are the same for every row it transforms, but 31 + 32 complex values do not fit in
// the register file next to the FFT working set and the MRC accumulators, so the kernels used to re-read them from a
// shared-memory table (or regenerate them by a recurrence) for every row -- on the very pipes that bound them.
// Blackwell's tensor memory is a third on-chip store with its own data path: 128 lanes x 512 32-bit columns per SM,
// lane 32*(warp % 4) + l private to thread l of the warp when accessed with the 32x32b shape.  Measured on B200
// (tools/ubench_tmem.cu, profiles/r02_ubench_tmem.txt): next to a saturated shared-memory port, fetching 16 complex
// constants per row costs +24 % from shared memory and +1.5 % from tensor memory.
// Each CTA (exactly 4 warps) allocates kTmemCols columns once and frees them at exit.
__device__ __forceinline__ uint32_t tmem_alloc_cols(uint32_t* s_slot, int n_cols_pow2, int warp)
{
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_slot)), "r"(n_cols_pow2) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    return *s_slot + (((uint32_t)(warp & 3) * 32u) << 16);  // this warp's lane quarter
}
__device__ __forceinline__ void tmem_free_cols(uint32_t base, int n_cols_pow2, int warp)
{
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(n_cols_pow2) : "memory");
}
// 4 complex values -> columns [col, col + 8) of the calling thread's lane
__device__ __forceinline__ void tmem_store4(uint32_t taddr, int col, const float2 (&v)[4])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr + (uint32_t)col),
                 "r"(__float_as_uint(v[0].x)), "r"(__float_as_uint(v[0].y)), "r"(__float_as_uint(v[1].x)), "r"(__float_as_uint(v[1].y)),
                 "r"(__float_as_uint(v[2].x)), "r"(__float_as_uint(v[2].y)), "r"(__float_as_uint(v[3].x)), "r"(__float_as_uint(v[3].y))
                 : "memory");
}
__device__ __forceinline__ void tmem_store_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 8 complex values <- columns [col, col + 16); returns after the load has landed (the registers pass through the
// wait so that no use can be scheduled ahead of it)
__device__ __forceinline__ void tmem_load8(uint32_t taddr, int col, float2 (&v)[8])
{
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr + (uint32_t)col));
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
}

template <class PL>
__device__ __forceinline__ void team_sync(int team)
{
    if constexpr (PL::T <= 32) {
        __syncwarp();
    } else if constexpr (PL::TEAMS == 1) {
        __syncthreads();
    } else {
        asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "n"(PL::T) : "memory");
    }
}

// Hard decision, Gray-mapped square QAM (3GPP TS 38.211 5.1.3-5.1.5, unit average
// power); identical constants and comparisons to oracle/cpuls_oracle.c demap_one().
__device__ __forceinline__ unsigned demap_symbol(float re, float im, int qam_bits)
{
    const float t16 = (float)0.6324555320336759;
    const float t4 = (float)0.6172133998483676;
    const float t2 = (float)0.3086066999241838;
    unsigned v = 0;
    const float are = fabsf(re), aim = fabsf(im);
    if (re < 0.0f) v |= 1u;
    if (im < 0.0f) v |= 2u;
    if (qam_bits == 4) {
        if (are > t16) v |= 4u;
        if (aim > t16) v |= 8u;
    } else if (qam_bits == 6) {
        if (are > t4) v |= 4u;
        if (aim > t4) v |= 8u;
        if (fabsf(__fsub_rn(are, t4)) > t2) v |= 16u;
        if (fabsf(__fsub_rn(aim, t4)) > t2) v |= 32u;
    }
    return v;
}

template <class PL>
__device__ __forceinline__ void row_load(float2 (&v)[PL::P], const float2* __restrict__ x, int t)
{
#pragma unroll
    for (int n1 = 0; n1 < PL::P; ++n1) {
        v[n1] = ld_stream(x + n1 * PL::T + t);
    }
}

// the same for rows that are only 4-byte aligned: two 32-bit loads per sample
template <class PL>
__device__ __forceinline__ void row_load_align4(float2 (&v)[PL::P], const float2* __restrict__ x, int t)
{
    const float* xs = reinterpret_cast<const float*>(x);
#pragma unroll
    for (int n1 = 0; n1 < PL::P; ++n1) {
        const float* q = xs + 2 * (n1 * PL::T + t);
        asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v[n1].x) : "l"(q));
        asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v[n1].y) : "l"(q + 1));
    }
}

// Max-log LLRs of the Gray-mapped square QAM of demap_symbol(), the usual piecewise-linear form:
//   bit 0/1 (sign bits):       4a*rho * re|im
//   16-QAM bit 2/3:            4a*rho * (2a - |re|im|)
//   64-QAM bit 2/3, bit 4/5:   4a*rho * (4a - |.|),  4a*rho * (2a - ||.| - 4a|)
// a = 1/sqrt(2), 1/sqrt(10), 1/sqrt(42); rho = sum|H|^2 / noise_var is the post-MRC SNR scale.
// Same constants and operation order as oracle/cpuls_oracle.c soft_one().
template <int B>
__device__ __forceinline__ void soft_symbol(float re, float im, float rho, float* out)
{
    constexpr float a = (B == 2) ? (float)0.7071067811865476 : (B == 4) ? (float)0.31622776601683794 : (float)0.1543033499620919;
    const float g = __fmul_rn(4.0f * a, rho);
    out[0] = __fmul_rn(g, re);
    out[1] = __fmul_rn(g, im);
    if (B == 4) {
        out[2] = __fmul_rn(g, __fsub_rn(2.0f * a, fabsf(re)));
        out[3] = __fmul_rn(g, __fsub_rn(2.0f * a, fabsf(im)));
    } else if (B == 6) {
        out[2] = __fmul_rn(g, __fsub_rn(4.0f * a, fabsf(re)));
        out[3] = __fmul_rn(g, __fsub_rn(4.0f * a, fabsf(im)));
        out[4] = __fmul_rn(g, __fsub_rn(2.0f * a, fabsf(__fsub_rn(fabsf(re), 4.0f * a))));
        out[5] = __fmul_rn(g, __fsub_rn(2.0f * a, fabsf(__fsub_rn(fabsf(im), 4.0f * a))));
    }
}

// One N-point forward DFT of the row whose samples are already in `v` (v[n1] = x[n1*T + t],
// CP skipped); the team's P*T outputs are handed to `sink(slot, bin, value)` where slot in
// [0,P) is the thread-local accumulator index and bin = c + (N/RL)*j is the FFT bin.
// If x_next != nullptr the next row is loaded into `v` as soon as stage 1 has consumed it,
// so its HBM latency hides behind stage 2/3 and the MRC of this row (register prefetch).
// Last stage of the shuffle-stage plans for a batch of JB register pairs: the radix-SH transform over the SH adjacent
// lanes q = lane % SH.  keep[i] / send[i] are registers 2j / 2j+1 of the stage-2 transform (already twiddled; which
// k2 they hold depends on the lane, see Plan::stage1_sign); A[i] / B[i] are the outputs of slots 2j / 2j+1, each
// times the slot's unit factor (Plan::unit_mul).  All shuffles of a round are issued back to back so that their
// latencies overlap.
//   SH = 2: one round, partner lane ^ 1:            A = keep + r, B = keep - r
//   SH = 4: decimation in time over q = 2*q1 + q0.  Round 1, partner lane ^ 2 (same q0):
//             p = keep + s0*r1, m = keep - s0*r1, s0 = +1 on even lanes, -1 on odd lanes
//             (even lanes: p = E+, m = sigma1*E-; odd lanes: p = sigma1*O-, m = O+; sigma1 = +-1 by q1), so that every
//             lane keeps p and sends m; round 2, partner lane ^ 1:
//             even lanes A = p + r2 = X[k3 = 0], B = p - r2 = X[2];  odd lanes A = p + i*r2 = i*sigma1*X[1],
//             B = p - i*r2 = -i*sigma1*X[3]
template <int SH, int JB>
__device__ __forceinline__ void sh_radix_batch(const float2 (&keep)[JB], const float2 (&send)[JB], int q, float2 (&A)[JB], float2 (&B)[JB])
{
    if constexpr (SH == 2) {
        float2 r1[JB];
#pragma unroll
        for (int i = 0; i < JB; ++i) {
            r1[i].x = __shfl_xor_sync(0xffffffffu, send[i].x, 1);
            r1[i].y = __shfl_xor_sync(0xffffffffu, send[i].y, 1);
        }
#pragma unroll
        for (int i = 0; i < JB; ++i) {
            A[i] = cadd(keep[i], r1[i]);
            B[i] = csub(keep[i], r1[i]);
        }
    } else {
        const bool odd = (q & 1) != 0;
        const float s0 = odd ? -1.f : 1.f;
        const float2 sp = make_float2(s0, s0), sm = make_float2(-s0, -s0);
        float2 r1[JB], pp[JB], mm[JB], r2[JB];
#pragma unroll
        for (int i = 0; i < JB; ++i) {
            r1[i].x = __shfl_xor_sync(0xffffffffu, send[i].x, 2);
            r1[i].y = __shfl_xor_sync(0xffffffffu, send[i].y, 2);
        }
#pragma unroll
        for (int i = 0; i < JB; ++i) {
            pp[i] = __ffma2_rn(r1[i], sp, keep[i]);
            mm[i] = __ffma2_rn(r1[i], sm, keep[i]);
        }
#pragma unroll
        for (int i = 0; i < JB; ++i) {
            r2[i].x = __shfl_xor_sync(0xffffffffu, mm[i].x, 1);
            r2[i].y = __shfl_xor_sync(0xffffffffu, mm[i].y, 1);
        }
#pragma unroll
        for (int i = 0; i < JB; ++i) {
            // odd lanes: i*r2 = (-r2.y, r2.x); the negation rides on the select, so both kinds of lane finish with
            // the same two packed adds and no per-lane constant pair has to be kept (or rebuilt) in registers
            const float2 rr = make_float2(odd ? -r2[i].y : r2[i].x, odd ? r2[i].x : r2[i].y);
            A[i] = cadd(pp[i], rr);
            B[i] = csub(pp[i], rr);
        }
    }
}

constexpr int kShBatch = 4;  // register pairs per shuffle batch (= one 8-slot chunk of the Hconj ring)

// twiddles W_T^(q*k2) of the 2*JB registers of batch jb.  Register r of lane position q holds k2 = brev(r & ~1) +
// 16*(hi ^ (r & 1)), hi = the high bit of q; the table is laid out per lane position, [16 register pairs][SH] entries of
// (twiddle of register 2j, twiddle of register 2j+1), so a pair is ONE 128-bit load whose SH distinct addresses per
// warp are broadcast (one shared-memory wavefront instead of four for two 64-bit loads).  twq = table + 2*q.
template <int SH, int JB>
__device__ __forceinline__ void sh_load_twiddles(float2 (&tw)[2 * JB], const float2* twq, int jb)
{
#pragma unroll
    for (int i = 0; i < JB; ++i) {
        const float2* src = twq + (JB * jb + i) * SH * 2;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(tw[2 * i].x), "=f"(tw[2 * i].y), "=f"(tw[2 * i + 1].x), "=f"(tw[2 * i + 1].y)
                     : "r"(smem_u32(src)));
    }
}

// stage-2 operands of thread (k1, q) of a shuffle-stage plan: element n2*SH + q of tile row k1, n2 = 0..31, out of the
// swizzled tile (Plan::at): column SH*(n2 ^ g) + q with g = k1 mod G, G = 16/SH.  Writing n2 = G*m + i, the address is
// (row + q + SH*(i ^ g)) + 16*m: G base pointers and compile-time offsets.
template <class PL>
__device__ __forceinline__ void sh_stage2_read(float2 (&u)[32], const float2* __restrict__ tile, int k1, int q)
{
    constexpr int SH = PL::SH, G = 16 / SH;
    const int g = k1 % G;
    const float2* row = tile + k1 * PL::ROW + q;
#pragma unroll
    for (int i = 0; i < G; ++i) {
        const float2* base = row + SH * (i ^ g);
#pragma unroll
        for (int m = 0; m < 32 / G; ++m) u[G * m + i] = base[16 * m];
    }
}

// writes the P stage-1 factors of thread t (k1 = 0: the bare sign, else the signed table entry) to columns [0, 2P)
template <class PL>
__device__ __forceinline__ void tmem_fill_stage1(uint32_t tmem, const float2* __restrict__ table, int t)
{
    const float sg = PL::stage1_sign(t);
#pragma unroll
    for (int c = 0; c < PL::P / 4; ++c) {
        float2 w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = 4 * c + i;
            w[i] = (r == 0) ? make_float2(sg, 0.f) : table[(r - 1) * PL::T + t];  // (the table carries the sign)
        }
        tmem_store4(tmem, 8 * c, w);
    }
}

// Zero-instruction scheduling fence for register values: everything v[] depends on is computed before this point and
// nothing that uses v[] afterwards is started ahead of it.  Used to keep arithmetic on the near side of a wait (the
// compiler may move plain arithmetic across a volatile asm, e.g. sink a transform below an mbarrier wait and so
// shorten the time the awaited copy has to land).
template <int NV>
__device__ __forceinline__ void pin_values(float2 (&v)[NV])
{
    static_assert(NV % 8 == 0, "groups of eight");
#pragma unroll
    for (int i = 0; i < NV; i += 8)
        asm volatile("" : "+f"(v[i].x), "+f"(v[i].y), "+f"(v[i + 1].x), "+f"(v[i + 1].y), "+f"(v[i + 2].x), "+f"(v[i + 2].y), "+f"(v[i + 3].x),
                          "+f"(v[i + 3].y), "+f"(v[i + 4].x), "+f"(v[i + 4].y), "+f"(v[i + 5].x), "+f"(v[i + 5].y), "+f"(v[i + 6].x),
                          "+f"(v[i + 6].y), "+f"(v[i + 7].x), "+f"(v[i + 7].y));
}

struct NoHook {
    __device__ __forceinline__ void operator()() const {}
};

// `after_reads` (two-stage plans) runs once the last-stage operands have been read from the tile, before the
// last-stage arithmetic: from then on this row no longer needs the tile.
template <class PL, class Sink, class Hook = NoHook>
__device__ __forceinline__ void row_fft(float2 (&v)[PL::P], const float2* __restrict__ x_next,
                                        float2* __restrict__ tile, const float2* __restrict__ s_tw1,
                                        const float2* __restrict__ s_tw2, int t, int team, Sink&& sink,
                                        uint32_t tmem_tw = 0, Hook&& after_reads = Hook())
{
    constexpr int P = PL::P, T = PL::T, ROW = PL::ROW, R2 = PL::R2, R3 = PL::R3;
    fft_reg<P>(v);
    if (PL::TW_TMEM && tmem_tw != 0) {
        // inter-stage twiddles from the thread's tensor-memory lane: columns [0, 2P) hold stage1_sign(t) * W_N^(t*k1),
        // k1 = 0..P-1 (entry 0 is the bare sign), written once per kernel by tmem_fill_stage1
#pragma unroll
        for (int c = 0; c < P / 8; ++c) {
            float2 w[8];
            tmem_load8(tmem_tw, 16 * c, w);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k1 = 8 * c + i;
                float2 val = v[brev<P>(k1)];
                if (k1 > 0 || PL::SH > 1) val = cmul(val, w[i]);
                tile[PL::at(k1, t)] = val;
            }
        }
    } else {
    // Inter-stage twiddles W_N^(t*k1) come from the shared table.  They are fetched in chunks of
    // TWC, one chunk ahead of the multiplies that use them, through volatile loads fenced with
    // compiler barriers: left to itself ptxas (168-register budget) sinks every twiddle load to
    // just before its multiply and exposes the ~30-cycle shared-memory latency 31 times per row.
    constexpr int TWC = PL::TW_CHUNK;
    static_assert(P % TWC == 0, "chunk must divide P");
    float2 twa[TWC], twb[TWC];
#pragma unroll
    for (int j = 0; j < TWC; ++j) twa[j] = (j == 0) ? make_float2(1.f, 0.f) : lds_volatile(s_tw1 + (j - 1) * T + t);
    asm volatile("" ::: "memory");
#pragma unroll
    for (int c = 0; c < P / TWC; ++c) {
        if (c + 1 < P / TWC) {
#pragma unroll
            for (int j = 0; j < TWC; ++j) twb[j] = lds_volatile(s_tw1 + ((c + 1) * TWC + j - 1) * T + t);
        }
        asm volatile("" ::: "memory");
#pragma unroll
        for (int j = 0; j < TWC; ++j) {
            const int k1 = c * TWC + j;
            float2 val = v[brev<P>(k1)];
            if (k1 > 0) {
                val = cmul(val, twa[j]);  // (shuffle-stage plans: the table carries stage1_sign(t))
            } else if (PL::SH > 1) {
                const float sg = PL::stage1_sign(t);
                val = __fmul2_rn(val, make_float2(sg, sg));
            }
            tile[PL::at(k1, t)] = val;
        }
        asm volatile("" ::: "memory");
#pragma unroll
        for (int j = 0; j < TWC; ++j) twa[j] = twb[j];
    }
    }
    if (x_next != nullptr) row_load<PL>(v, x_next, t);
    team_sync<PL>(team);
    if constexpr (PL::SH > 1) {
        // ---- shuffle-stage plans: N = 32 * 32 * SH.  Thread (k1, q), q = lane % SH, transforms the 32 samples
        // t2 = n2*SH + q of row k1 of the tile; the remaining radix-SH stage over q runs across the SH adjacent lanes.
        // A plain transpose would make every lane choose which half of its registers to send (selects); instead the
        // sign trick of Plan::stage1_sign leaves U[kk + 16*hi] in register 2j ("keep") and U[kk + 16*(1-hi)] in
        // 2j+1 ("send"), hi = the high bit of q, so the choice is the same instruction in every lane.
        constexpr int SH = PL::SH;
        const int lane = t & 31;
        const int q = lane % SH;
        const int k1 = lane / SH + (32 / SH) * (t >> 5);
        float2 u[32];
        sh_stage2_read<PL>(u, tile, k1, q);
        after_reads();  // the tile is free from here on
        fft_reg<32>(u);
        // twiddles W_T^(q*k2), fetched one batch ahead of their multiplies; then the cross-lane radix-SH stage
        constexpr int JB = kShBatch;
        const float2* twq = s_tw2 + 2 * q;
        float2 tw[2 * JB], twn[2 * JB];
        sh_load_twiddles<SH, JB>(tw, twq, 0);
#pragma unroll
        for (int jb = 0; jb < 16 / JB; ++jb) {
            if (jb + 1 < 16 / JB) sh_load_twiddles<SH, JB>(twn, twq, jb + 1);
            asm volatile("" ::: "memory");
            float2 keep[JB], send[JB], A[JB], B[JB];
#pragma unroll
            for (int i = 0; i < JB; ++i) {
                keep[i] = cmul(u[2 * (JB * jb + i)], tw[2 * i]);
                send[i] = cmul(u[2 * (JB * jb + i) + 1], tw[2 * i + 1]);
            }
            sh_radix_batch<SH, JB>(keep, send, q, A, B);
#pragma unroll
            for (int i = 0; i < JB; ++i) {
                const int sl = 2 * (JB * jb + i);
                sink(sl, PL::bin_of(sl, t), A[i]);
                sink(sl + 1, PL::bin_of(sl + 1, t), B[i]);
            }
#pragma unroll
            for (int i = 0; i < 2 * JB; ++i) tw[i] = twn[i];
        }
    } else {
#pragma unroll
    for (int i = 0; i < PL::NB2; ++i) {
        const int b = t + T * i;
        const int k1 = b % P, m2 = b / P;
        float2 u[R2];
        float2* col = tile + k1 * ROW + m2;
#pragma unroll
        for (int n2 = 0; n2 < R2; ++n2) u[n2] = col[n2 * R3];
        if constexpr (R3 == 1) {
            if (i == PL::NB2 - 1) after_reads();
        }
        fft_reg<R2>(u);
        if constexpr (R3 == 1) {
#pragma unroll
            for (int k2 = 0; k2 < R2; ++k2) sink(i * R2 + k2, b + (PL::N / R2) * k2, u[brev<R2>(k2)]);
        } else {
            // second-level twiddles W_T^(m2*k2): same chunk-ahead fetch as the first level
            constexpr int C2 = (R2 >= 8) ? PL::TW_CHUNK : R2;
            float2 wa[C2], wb[C2];
#pragma unroll
            for (int j = 0; j < C2; ++j) wa[j] = (j == 0) ? make_float2(1.f, 0.f) : lds_volatile(s_tw2 + (j - 1) * R3 + m2);
            asm volatile("" ::: "memory");
#pragma unroll
            for (int c = 0; c < R2 / C2; ++c) {
                if (c + 1 < R2 / C2) {
#pragma unroll
                    for (int j = 0; j < C2; ++j) wb[j] = lds_volatile(s_tw2 + ((c + 1) * C2 + j - 1) * R3 + m2);
                }
                asm volatile("" ::: "memory");
#pragma unroll
                for (int j = 0; j < C2; ++j) {
                    const int k2 = c * C2 + j;
                    float2 val = u[brev<R2>(k2)];
                    if (k2 > 0) val = cmul(val, wa[j]);
                    col[k2 * R3] = val;
                }
                asm volatile("" ::: "memory");
#pragma unroll
                for (int j = 0; j < C2; ++j) wa[j] = wb[j];
            }
        }
    }
    if constexpr (R3 > 1 && PL::X_TMA) {
        // bulk-copy plans: read ALL last-stage operands first so that the tile is free for the next row's copy
        // while the R3-point butterflies and the sink (MRC) run
        team_sync<PL>(team);
        float2 w[PL::NB3][R3];
#pragma unroll
        for (int i = 0; i < PL::NB3; ++i) {
            const int c = t + T * i;
            const float2* src = tile + (c % P) * ROW + (c / P) * R3;
#pragma unroll
            for (int m2 = 0; m2 < R3; ++m2) w[i][m2] = src[m2];
        }
        after_reads();
#pragma unroll
        for (int i = 0; i < PL::NB3; ++i) {
            const int c = t + T * i;
            fft_reg<R3>(w[i]);
#pragma unroll
            for (int k3 = 0; k3 < R3; ++k3) sink(i * R3 + k3, c + (PL::N / R3) * k3, w[i][brev<R3>(k3)]);
        }
    } else if constexpr (R3 > 1) {
        team_sync<PL>(team);
#pragma unroll
        for (int i = 0; i < PL::NB3; ++i) {
            const int c = t + T * i;
            const int k1 = c % P, k2 = c / P;
            float2 w[R3];
            const float2* src = tile + k1 * ROW + k2 * R3;
#pragma unroll
            for (int m2 = 0; m2 < R3; ++m2) w[m2] = src[m2];
            fft_reg<R3>(w);
#pragma unroll
            for (int k3 = 0; k3 < R3; ++k3) sink(i * R3 + k3, c + (PL::N / R3) * k3, w[brev<R3>(k3)]);
        }
    }
    }  // plans without a shuffle stage
    if constexpr (PL::NBUF == 1) team_sync<PL>(team);
}

// Bit packing of one row by a team: the K demapped symbols in s_idx, b bits each, as one bit stream (bit j of the row =
// bit j % b of symbol j / b) into bit j % 8 of byte j / 8.  Nothing is stored unless `store`.
template <class PL>
__device__ __forceinline__ void pack_bits(const uint8_t* s_idx, uint8_t* bits_row, int row_bytes, int b, bool store, int t)
{
    constexpr int K = PL::N - 1;
    for (int byte = t; byte < row_bytes; byte += PL::T) {
        unsigned v8 = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int pos = byte * 8 + q;
            const int sym = pos / b, bit = pos - sym * b;
            if (sym < K) v8 |= ((s_idx[sym] >> bit) & 1u) << q;
        }
        if (store) bits_row[byte] = (uint8_t)v8;
    }
}

// Epilogue of one (frame, data symbol) held by a team: normalise (cpuLS.hpp:364-367), reorder to
// ascending frequency (cpuLS.hpp:135-149), demap, pack, optional LLRs.  acc[sl] is the MRC sum of
// the bin the thread owns in slot sl; e_row[bin - 1] = sum_a |H|^2 (global, or shared when
// E_SHARED).  Specialised on the QAM order so the demapper and the bit packing are straight-line
// code.  s_idx: K bytes of team-private shared memory (aliases the team's tile).
template <class PL, bool E_SHARED, bool E_CG = false>
__device__ __forceinline__ void mrc_finish(const KernelParams& p, const float2 (&acc)[PL::P], const float* __restrict__ e_row,
                                           int f, int s, uint8_t* s_idx, bool valid, int t, int team)
{
    constexpr int N = PL::N, P = PL::P, K = N - 1;
    float2* out_row = p.combined + ((long long)f * p.n_sym_work + s) * K;
    uint8_t* bits_row = p.bits ? p.bits + ((long long)f * p.n_sym_work + s) * p.bits_row_bytes : nullptr;
    float* llr_row = p.llr ? p.llr + ((long long)f * p.n_sym_work + s) * K * p.qam_bits : nullptr;
    auto finish = [&](auto bconst) {
        constexpr int b = decltype(bconst)::value;
        float einv[P];
#pragma unroll
        for (int sl = 0; sl < P; ++sl) {
            const int bin = PL::bin_of(sl, t);
            const int idx = bin > 0 ? bin - 1 : 0;
            einv[sl] = E_SHARED ? e_row[idx] : (E_CG ? __ldcg(e_row + idx) : __ldg(e_row + idx));  // E_CG: written during this launch
        }
        team_sync<PL>(team);  // everyone is done reading the last tile before it is reused
#pragma unroll
        for (int sl = 0; sl < P; ++sl) {
            const int bin = PL::bin_of(sl, t);
            if (bin > 0) {
                // one reciprocal, two multiplies (<= 2 ulp from the reference's two divisions,
                // far inside the 1e-5 parity tolerance)
                const float inv = __frcp_rn(einv[sl]);
                const float2 o = make_float2(acc[sl].x * inv, acc[sl].y * inv);
                const int pos = (bin < N / 2) ? (bin - 1 + N / 2) : (bin - N / 2);
                if (valid) out_row[pos] = o;
                s_idx[pos] = (uint8_t)demap_symbol(o.x, o.y, b);
                if (llr_row != nullptr && valid) {
                    float l[b];
                    soft_symbol<b>(o.x, o.y, __fmul_rn(einv[sl], p.inv_noise_var), l);
#pragma unroll
                    for (int q = 0; q < b; ++q) llr_row[pos * b + q] = l[q];
                }
            }
        }
        if (bits_row != nullptr) {
            team_sync<PL>(team);
            pack_bits<PL>(s_idx, bits_row, p.bits_row_bytes, b, valid, t);
        }
    };
    if (p.qam_bits == 2) finish(std::integral_constant<int, 2>{});
    else if (p.qam_bits == 4) finish(std::integral_constant<int, 4>{});
    else finish(std::integral_constant<int, 6>{});
}

// LS divide of the generic pilot paths (pilot kernel, one-launch kernel), per slot of the thread: the pilot value of
// the slot's bin (load) and 1/|X|^2 (recip), hoisted out of the per-element divide of cpuLS.hpp:240-241 (<= 1 ulp apart).
template <class PL>
struct LsDivide {
    float2 xp[PL::P];
    float xden[PL::P];
    __device__ __forceinline__ void load(const KernelParams& p, int sl, int t)
    {
        const int bin = PL::bin_of(sl, t);
        xp[sl] = p.pilot_bin[bin > 0 ? bin - 1 : 0];
    }
    __device__ __forceinline__ void recip(int sl) { xden[sl] = 1.0f / (xp[sl].x * xp[sl].x + xp[sl].y * xp[sl].y); }
    // the LS estimate H = Z / X of slot sl from its FFT output z (cpuLS.hpp:233-244); conj(H) is what gets stored
    // (:303-307), |H|^2 = energy(H) what gets summed (cpuLS.hpp:211-228)
    __device__ __forceinline__ float2 divide(int sl, float2 z) const
    {
        const float2 X = xp[sl];
        return make_float2((z.x * X.x + z.y * X.y) * xden[sl], (z.y * X.x - z.x * X.y) * xden[sl]);
    }
    static __device__ __forceinline__ float energy(float2 h) { return h.x * h.x + h.y * h.y; }
};

// XT (data mode of X_TMA plans): antenna rows come in by bulk copy.  A compile-time switch, not a test of p.x_tma inside the
// row loop: with both paths in one loop body ptxas schedules the common one 2 % slower (c2: 2.42 -> 2.36 ms per 256 frames).
template <class PL, int MODE, int MINB, bool XT = false>
__global__ void __launch_bounds__(PL::THREADS, MINB) lsmrc_kernel(const KernelParams p)
{
    constexpr int N = PL::N, P = PL::P, T = PL::T, K = N - 1;
    constexpr int PF_X = PL::PF_X, PF_H = PL::PF_H;
    extern __shared__ __align__(16) float2 smem[];
    float2* s_tw1 = smem;
    float2* s_tw2 = smem + PL::TW1;
    float2* s_hring = smem + PL::TWN;
    float2* s_tiles = smem + PL::TWN + PL::HRING;

    const int team = threadIdx.x / T;
    const int t = threadIdx.x % T;
    float2* my_tiles = s_tiles + team * PL::TEAM_STRIDE;

    if constexpr (MODE != MODE_ONESHOT) {  // (the one-shot mode issues its first row loads before this copy)
        for (int i = threadIdx.x; i < PL::TWN; i += PL::THREADS) smem[i] = p.twiddles[i];
        __syncthreads();
    }

    if constexpr (MODE == MODE_FFT) {
        // stand-alone batched transform (gpuLS::batchedFFT, gpuLS.cu:343-349): p.rx holds
        // p.n_frames rows of N samples (row stride p.ant_stride), transformed in place into
        // p.combined (may alias p.rx: a team has its whole row in registers before it stores)
        const int n_rows = p.n_frames;
        for (int row0 = blockIdx.x * PL::TEAMS; row0 < n_rows; row0 += gridDim.x * PL::TEAMS) {
            const int row_raw = row0 + team;
            const bool ok = row_raw < n_rows;
            const int row = ok ? row_raw : n_rows - 1;
            float2 v[P];
            row_load<PL>(v, p.rx + (long long)row * p.ant_stride + p.cp, t);
            float2* out = p.combined + (long long)row * N;
            team_sync<PL>(team);
            row_fft<PL>(v, nullptr, my_tiles, s_tw1, s_tw2, t, team, [&](int sl, int bin, float2 y) {
                if (ok) out[bin] = PL::unfix(sl, t, y);
            });
            team_sync<PL>(team);
        }
    } else if constexpr (MODE == MODE_PILOT) {
        // Virtual CTA (c, g): frames [c*fpc, (c+1)*fpc), antenna group g of n_groups.  Each of the fpc frames
        // gets tpf = TEAMS/fpc teams, which share the antennas of the group round-robin.  fpc > 1
        // (several frames per CTA, only with n_groups == 1) keeps all teams busy when a frame has
        // fewer antennas than the CTA has teams.  A CTA strides over the virtual CTAs (grid = at most one
        // resident wave), so the twiddle copy and the pilot reciprocals below are paid once per CTA.
        const int fpc = p.frames_per_cta;
        const int tpf = PL::TEAMS / fpc;
        const int lf = team / tpf, tj = team % tpf;
        LsDivide<PL> ls;
#pragma unroll
        for (int sl = 0; sl < P; ++sl) {
            ls.load(p, sl, t);
            ls.recip(sl);
        }
        const int n_virtual = ((p.n_frames + fpc - 1) / fpc) * p.n_groups;
        for (int vb = blockIdx.x; vb < n_virtual; vb += gridDim.x) {
        const int cta_f0 = (vb / p.n_groups) * fpc;
        const int g = vb % p.n_groups;
        const bool f_ok = lf < fpc && cta_f0 + lf < p.n_frames;
        const int f = f_ok ? cta_f0 + lf : p.n_frames - 1;
        const float2* x0 = p.rx + (long long)f * p.frame_stride + (long long)p.first_sym * p.sym_stride + p.cp;
        float2* hw_frame = p.hwork + (long long)f * p.n_ant * N;
        float2* hc_frame = p.hconj ? p.hconj + (long long)f * p.n_ant * K : nullptr;
        float e[P];
#pragma unroll
        for (int sl = 0; sl < P; ++sl) e[sl] = 0.f;
        const int per_iter = p.n_groups * tpf;
        const int n_iter = (p.n_ant + per_iter - 1) / per_iter;
        for (int it = 0; it < n_iter; ++it) {
            const int a_raw = (it * p.n_groups + g) * tpf + tj;
            const bool a_ok = f_ok && a_raw < p.n_ant;
            const int a = a_raw < p.n_ant ? a_raw : p.n_ant - 1;
            float2* tile = my_tiles + (PL::NBUF == 2 ? (it & 1) * PL::TILE : 0);
            float2* hw_row = hw_frame + (long long)a * N;
            float2* hc_row = hc_frame ? hc_frame + (long long)a * K : nullptr;
            float2 v[P];
            row_load<PL>(v, x0 + (long long)a * p.ant_stride, t);
            if (a_raw + per_iter < p.n_ant)  // this team's next antenna: pull its row into L2 meanwhile
                prefetch_row<T, false>(x0 + (long long)(a_raw + per_iter) * p.ant_stride, N, t);
            row_fft<PL>(v, nullptr, tile, s_tw1, s_tw2, t, team,
                        [&](int sl, int bin, float2 z) {
                            const float2 H = ls.divide(sl, z);
                            if (a_ok) {
                                // (shuffle-stage plans: z carries the unit factor of its slot, and so does the hc the
                                // data kernel will multiply its equally factored outputs with; the exported copy is exact)
                                const float2 hc = (bin > 0) ? make_float2(H.x, -H.y) : make_float2(0.f, 0.f);
                                hw_row[PL::hpos(sl, t, bin)] = hc;
                                if (bin > 0) {
                                    if (hc_row) hc_row[bin - 1] = PL::refix(sl, t, hc);
                                    e[sl] += ls.energy(H);
                                }
                            }
                        });
        }
        // deterministic cross-team sum of the energy partials, then cross-group by the last CTA
        __syncthreads();
        float* s_e = reinterpret_cast<float*>(s_tiles);  // [TEAMS][N]
#pragma unroll
        for (int sl = 0; sl < P; ++sl) {
            const int bin = PL::bin_of(sl, t);
            s_e[team * N + bin] = e[sl];
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < fpc * K; idx += PL::THREADS) {
            const int l2 = idx / K, bin = 1 + idx % K;
            const int f2 = cta_f0 + l2;
            if (f2 >= p.n_frames) break;
            const float* src = s_e + (l2 * tpf) * N + bin;
            float acc = src[0];
            for (int tm = 1; tm < tpf; ++tm) acc += src[tm * N];
            float* dst = (p.n_groups == 1) ? (p.hsqrd + (long long)f2 * K - 1) : (p.epart + ((long long)f2 * p.n_groups + g) * N);
            dst[bin] = acc;
        }
        if (p.n_groups > 1) {  // (fpc == 1 here)
            __shared__ unsigned int s_last;
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0) {
                const unsigned int prev = atomicAdd(p.counters + cta_f0, 1u);
                s_last = (prev == (unsigned)p.n_groups - 1u);
                if (s_last) p.counters[cta_f0] = 0u;  // self-reset for the next launch
            }
            __syncthreads();
            if (s_last) {
                __threadfence();
                const float* ep = p.epart + (long long)cta_f0 * p.n_groups * N;
                for (int bin = 1 + threadIdx.x; bin < N; bin += PL::THREADS) {
                    float acc = __ldcg(ep + bin);
                    for (int gg = 1; gg < p.n_groups; ++gg) acc += __ldcg(ep + (long long)gg * N + bin);
                    p.hsqrd[(long long)cta_f0 * K + bin - 1] = acc;
                }
            }
        }
        __syncthreads();  // the partial-energy buffer aliases the tiles of the next virtual CTA
        }  // virtual CTAs
    } else if constexpr (MODE == MODE_ONESHOT) {
        // Whole frames in ONE launch, for calls that are launch-latency bound (a single small frame,
        // BASELINE config c5): CTA (f, g) first estimates the channel of frame f itself -- all its
        // teams share the A pilot rows, conj(H) and sum|H|^2 stay in shared memory -- and then
        // combines its own `slots` data symbols against them.  Every CTA of a frame repeats the
        // pilot work (1/S of the frame, a round or two of row FFTs) in exchange for dropping the
        // second launch and the global round trip of H; CTA g == 0 also writes H to global memory
        // for callers that read it back.  The host picks this mode only when the whole batch is
        // one partial wave of CTAs and A*N conj(H) values fit in shared memory.
        float2* s_h = s_tiles + PL::TEAMS * PL::TEAM_STRIDE;                     // [A][N]
        float* s_esum = reinterpret_cast<float*>(s_h + (size_t)p.n_ant * N);     // [N], entry 0 unused
        const int AS = p.ant_split;           // teams sharing one (frame, symbol)
        const int slots = PL::TEAMS / AS;     // data symbols per CTA
        const int aj = team % AS;
        const int groups = (p.n_sym_work + slots - 1) / slots;
        const int f = blockIdx.x / groups;
        const int g = blockIdx.x % groups;
        const bool writer = (g == 0);
        int s = g * slots + team / AS;
        bool valid = s < p.n_sym_work;
        if (!valid) s = p.n_sym_work - 1;
        // symbol 0 of a frame = pilot, data from p.first_sym
        const bool ring = p.split_sym != 0x7fffffff;
        auto sym_ptr = [&](int sym) -> const float2* {
            if (!ring) return p.rx + (long long)f * p.frame_stride + (long long)sym * p.sym_stride + p.cp;
            const long long slot = (long long)f * (p.first_sym + p.n_sym_work) + sym;  // ring slot of this symbol
            return (slot < p.split_sym ? p.rx + slot * p.sym_stride : p.rx2 + (slot - p.split_sym) * p.sym_stride) + p.cp;
        };
        const float2* xf = sym_ptr(0);
        const float2* xd = sym_ptr(p.first_sym + s);

        // issue every load the first rounds need before anything waits: pilot row, first data row
        // (registers when they are cheap, L2 otherwise), pilot values, twiddles
        constexpr bool EARLY = (P <= 16);
        float2 v[P];
        float2 vd[EARLY ? P : 1];
        auto load_row = [&](auto& dst, const float2* src) {
            if (p.rx_align4) row_load_align4<PL>(dst, src, t);
            else row_load<PL>(dst, src, t);
        };
        {
            const int a0 = team < p.n_ant ? team : p.n_ant - 1;
            load_row(v, xf + (long long)a0 * p.ant_stride);
            const int ad = aj < p.n_ant ? aj : p.n_ant - 1;
            if constexpr (EARLY) load_row(vd, xd + (long long)ad * p.ant_stride);
            else prefetch_row<T, false>(xd + (long long)ad * p.ant_stride, N, t);
        }
        float e[P];
        LsDivide<PL> ls;
#pragma unroll
        for (int sl = 0; sl < P; ++sl) {
            e[sl] = 0.f;
            ls.load(p, sl, t);
        }
        for (int i = threadIdx.x; i < PL::TWN; i += PL::THREADS) smem[i] = p.twiddles[i];
#pragma unroll
        for (int sl = 0; sl < P; ++sl) ls.recip(sl);
        __syncthreads();

        // ---- channel estimate (same arithmetic as MODE_PILOT with one antenna group) ----
        float2* hw_frame = p.hwork + (long long)f * p.n_ant * N;
        float2* hc_frame = p.hconj ? p.hconj + (long long)f * p.n_ant * K : nullptr;
        const int n_iter = (p.n_ant + PL::TEAMS - 1) / PL::TEAMS;
        for (int it = 0; it < n_iter; ++it) {
            const int a_raw = it * PL::TEAMS + team;
            const bool a_ok = a_raw < p.n_ant;
            const int a = a_ok ? a_raw : p.n_ant - 1;
            float2* tile = my_tiles + (PL::NBUF == 2 ? (it & 1) * PL::TILE : 0);
            if (it > 0) load_row(v, xf + (long long)a * p.ant_stride);
            float2* sh_row = s_h + (size_t)a * N;
            float2* hw_row = hw_frame + (long long)a * N;
            float2* hc_row = hc_frame ? hc_frame + (long long)a * K : nullptr;
            row_fft<PL>(v, nullptr, tile, s_tw1, s_tw2, t, team, [&](int sl, int bin, float2 z) {
                const float2 H = ls.divide(sl, z);
                if (a_ok) {
                    const float2 hc = (bin > 0) ? make_float2(H.x, -H.y) : make_float2(0.f, 0.f);
                    sh_row[bin] = hc;  // (read back below by the same thread for the same slot: unit factors cancel)
                    if (writer) {
                        hw_row[PL::hpos(sl, t, bin)] = hc;
                        if (bin > 0 && hc_row) hc_row[bin - 1] = PL::refix(sl, t, hc);
                    }
                    if (bin > 0) e[sl] += ls.energy(H);
                }
            });
        }
        // sum the energy partials over the teams: the teams of a warp by shuffles, then the warps
        // (or the teams, when a team is a warp or more) through shared memory
        constexpr int TPW = (T < 32) ? 32 / T : 1;                        // teams per warp
        constexpr int NPART = (T < 32) ? (PL::THREADS + 31) / 32 : PL::TEAMS;
        if constexpr (TPW > 1) {
#pragma unroll
            for (int off = T; off < 32; off <<= 1) {
#pragma unroll
                for (int sl = 0; sl < P; ++sl) e[sl] += __shfl_xor_sync(0xffffffffu, e[sl], off);
            }
        }
        __syncthreads();
        float* s_e = reinterpret_cast<float*>(s_tiles);  // [NPART][N]
        if (team % TPW == 0) {
            const int part = team / TPW;
#pragma unroll
            for (int sl = 0; sl < P; ++sl) {
                const int bin = PL::bin_of(sl, t);
                s_e[part * N + bin] = e[sl];
            }
        }
        __syncthreads();
        for (int bin = 1 + threadIdx.x; bin < N; bin += PL::THREADS) {
            float acc = s_e[bin];
#pragma unroll
            for (int pt = 1; pt < NPART; ++pt) acc += s_e[pt * N + bin];
            s_esum[bin] = acc;
            if (writer) p.hsqrd[(long long)f * K + bin - 1] = acc;
        }
        __syncthreads();

        // ---- data symbols of this CTA against the shared-memory channel ----
        float2 acc[P];
#pragma unroll
        for (int sl = 0; sl < P; ++sl) acc[sl] = make_float2(0.f, 0.f);
        const int n_rounds = (p.n_ant + AS - 1) / AS;
        for (int rd = 0; rd < n_rounds; ++rd) {
            const int a_raw = rd * AS + aj;
            const bool a_ok = a_raw < p.n_ant;
            const int a = a_ok ? a_raw : p.n_ant - 1;
            float2* tile = my_tiles + (PL::NBUF == 2 ? (rd & 1) * PL::TILE : 0);
            if (EARLY && rd == 0) {
#pragma unroll
                for (int n1 = 0; n1 < P; ++n1) v[n1] = vd[EARLY ? n1 : 0];
            } else {
                load_row(v, xd + (long long)a * p.ant_stride);
            }
            if (a_raw + AS < p.n_ant) prefetch_row<T, false>(xd + (long long)(a_raw + AS) * p.ant_stride, N, t);
            const float2* h_row = s_h + (size_t)a * N;
            row_fft<PL>(v, nullptr, tile, s_tw1, s_tw2, t, team, [&](int sl, int bin, float2 y) {
                if (a_ok) acc[sl] = cmac(acc[sl], h_row[bin], y);
            });
        }
        if (AS > 1) {
            // add the antenna slices: teams that share a warp by shuffles, the rest through shared memory
            const int G = AS < TPW ? AS : TPW;  // teams combined inside a warp
            if constexpr (TPW > 1) {
                for (int off = T; off < T * G; off <<= 1) {
#pragma unroll
                    for (int sl = 0; sl < P; ++sl) {
                        acc[sl].x += __shfl_xor_sync(0xffffffffu, acc[sl].x, off);
                        acc[sl].y += __shfl_xor_sync(0xffffffffu, acc[sl].y, off);
                    }
                }
            }
            const int rem = AS / G;  // partial sums left per (frame, symbol)
            if (rem > 1) {
                float2* red = s_tiles;  // [TEAMS / G][P*T], aliases the tiles (all teams are past their last row)
                __syncthreads();
                if (team % G == 0) {
#pragma unroll
                    for (int sl = 0; sl < P; ++sl) red[((team / G) * P + sl) * T + t] = acc[sl];
                }
                __syncthreads();
                if (aj == 0) {
                    for (int jj = 1; jj < rem; ++jj) {
#pragma unroll
                        for (int sl = 0; sl < P; ++sl) acc[sl] = cadd(acc[sl], red[((team / G + jj) * P + sl) * T + t]);
                    }
                }
                __syncthreads();
            }
            valid = valid && (aj == 0);
        }
        mrc_finish<PL, true>(p, acc, s_esum + 1, f, s, reinterpret_cast<uint8_t*>(my_tiles), valid, t, team);
    } else {
        // Persistent CTAs: the grid is sized to the SM count and every CTA pulls work items from a
        // global ticket counter (dynamic, so faster SMs take more), so the twiddle table, the ring
        // barriers and the launch ramp are paid once per CTA instead of once per item.  Work item = TEAMS (frame, data symbol) pairs -- of one
        // frame when the Hconj ring is on -- one pair per team; each team loops over all antennas
        // and accumulates in registers.
        //
        // Hconj ring: stage R%H_STAGES holds the R-th row this CTA consumes (R counts across
        // items); full[] completes on the copy's bytes, empty[] when every team has consumed the
        // row.  Thread 0 keeps H_AHEAD rows in flight ahead of the row being consumed; a stage is
        // only refilled two rows after its last use, so the producer practically never waits on a
        // straggling team.
        __shared__ __align__(8) uint64_t bar_full[PL::H_STAGES], bar_empty[PL::H_STAGES];
        __shared__ __align__(8) uint64_t bar_x[PL::TEAMS];  // X_TMA: one per team, completes on the row's bytes
        uint32_t x_phase = 0;
        constexpr uint32_t ROW_BYTES = N * sizeof(float2);
        if constexpr (PL::H_RING) {
            if (threadIdx.x == 0) {
                for (int i = 0; i < PL::H_STAGES; ++i) {
                    mbar_init(&bar_full[i], 1);
                    mbar_init(&bar_empty[i], PL::TEAMS);
                }
                if constexpr (PL::X_TMA) {
                    for (int i = 0; i < PL::TEAMS; ++i) mbar_init(&bar_x[i], 1);
                }

                mbar_fence_init();
            }
            __syncthreads();
        }
        const int groups = (p.n_sym_work + PL::TEAMS - 1) / PL::TEAMS;
        const long long n_work = (long long)p.n_frames * p.n_sym_work;
        const int AS = PL::H_RING ? 1 : p.ant_split;     // teams sharing one (frame, symbol)
        const int slots = PL::TEAMS / AS;                // (frame, symbol) pairs per work item
        const int aj = team % AS;                        // this team's antenna slice
        const int n_items = PL::H_RING ? p.n_frames * groups : (int)((n_work + slots - 1) / slots);
        int rows_done = 0;  // ring rows consumed by this CTA so far

        // producer side of the ring: refill the stage of ring row R with Hconj row `row` of `src`
        auto ring_issue = [&](int R, const float2* src_row) {
            const int sr = R % PL::H_STAGES;
            const int use = R / PL::H_STAGES;
            if (use > 0) mbar_wait(&bar_empty[sr], (uint32_t)((use - 1) & 1));
            mbar_expect_tx(&bar_full[sr], ROW_BYTES);
            bulk_g2s(s_hring + sr * N, src_row, ROW_BYTES, &bar_full[sr]);
        };

        __shared__ uint32_t s_tmem;
        uint32_t tmem = 0;
        constexpr int kTmemCols = 2 * P;
        if constexpr (PL::TW_TMEM) {
            tmem = tmem_alloc_cols(&s_tmem, kTmemCols, (int)(threadIdx.x >> 5));
            tmem_fill_stage1<PL>(tmem, p.twiddles, t);
            tmem_store_wait();
        }
        __shared__ int s_item;
        for (;;) {
        if (threadIdx.x == 0) {
            const unsigned long long tk = atomicAdd(p.ticket, 1ULL);
            s_item = tk < (unsigned long long)n_items ? (int)tk : -1;
            if (s_item < 0) {
                // this CTA is done drawing; the last such CTA re-arms the counters for the next launch
                __threadfence();
                if (atomicAdd(p.ticket + 1, 1ULL) == (unsigned long long)gridDim.x - 1ULL) {
                    p.ticket[0] = 0ULL;
                    p.ticket[1] = 0ULL;
                }
            }
        }
        __syncthreads();
        const int item = s_item;
        __syncthreads();  // s_item is rewritten by thread 0 at the top of the next round
        if (item < 0) break;
        int f, s;
        bool valid;
        if constexpr (PL::H_RING) {
            f = item / groups;
            s = (item % groups) * PL::TEAMS + team;
            valid = s < p.n_sym_work;
            if (!valid) s = p.n_sym_work - 1;
        } else {
            long long work = (long long)item * slots + team / AS;
            valid = work < n_work;
            if (!valid) work = n_work - 1;
            f = (int)(work / p.n_sym_work);
            s = (int)(work % p.n_sym_work);
        }
        const float2* x0 = p.rx + (long long)f * p.frame_stride + (long long)(p.first_sym + s) * p.sym_stride + p.cp;
        const float2* hw_frame = p.hwork + (long long)f * p.n_ant * N;
        float2 acc[P];
#pragma unroll
        for (int sl = 0; sl < P; ++sl) acc[sl] = make_float2(0.f, 0.f);

        if constexpr (PL::H_RING) {
            if (threadIdx.x == 0) {
                for (int r = 0; r < PL::H_AHEAD && r < p.n_ant; ++r) ring_issue(rows_done + r, hw_frame + (long long)r * N);
            }
        }

        float2 v[P];
        if (PL::REG_PF != 0) row_load<PL>(v, x0 + (long long)(aj < p.n_ant ? aj : p.n_ant - 1) * p.ant_stride, t);  // this team's first antenna
        // XT: row a of this team's symbol arrives in the team's tile by bulk copy; row 0 is requested here,
        // row a+1 from inside row a (see the hook below).  (The launcher picks XT only when rows are 16-byte aligned.)
        static_assert(!XT || PL::X_TMA, "bulk-copied rows: X_TMA plans (whose teams never split a pair's antennas)");
        if (XT && t == 0) {
            fence_proxy_async();  // the tile doubled as the previous item's demap byte buffer
            mbar_expect_tx(&bar_x[team], ROW_BYTES);
            bulk_g2s(my_tiles, x0, ROW_BYTES, &bar_x[team]);
        }
        const int n_rounds = (p.n_ant + AS - 1) / AS;
        for (int rd = 0; rd < n_rounds; ++rd) {
            // antenna of this round; teams whose slice has run out redo the last antenna and drop the result
            const int a_raw = rd * AS + aj;
            const bool a_ok = a_raw < p.n_ant;
            const int a = a_ok ? a_raw : p.n_ant - 1;
            float2* tile = my_tiles + (PL::NBUF == 2 ? (rd & 1) * PL::TILE : 0);
            const float2* hw_row = hw_frame + (long long)a * N;
            if constexpr (PL::H_RING) {
                const int r = a + PL::H_AHEAD;
                if (threadIdx.x == 0 && r < p.n_ant) ring_issue(rows_done + r, hw_frame + (long long)r * N);
                __syncwarp();
            }
            const float2* x_next = nullptr;
            if (PL::REG_PF != 0) {
                if (a + AS < p.n_ant) x_next = x0 + (long long)(a + AS) * p.ant_stride;
            }
            if (XT) {
                mbar_wait(&bar_x[team], x_phase);
                x_phase ^= 1u;
#pragma unroll
                for (int n1 = 0; n1 < P; ++n1) v[n1] = tile[n1 * T + t];  // as the copy laid the row out: linear
                team_sync<PL>(team);  // every lane has its samples before stage 1 overwrites the tile
            } else if (PL::REG_PF == 0) {
                row_load<PL>(v, x0 + (long long)a * p.ant_stride, t);
            }
            // L2 prefetch: one row ahead of the demand loads, or one row ahead of the next bulk copy
            // (X_TMA plans whose rows are not 16-byte aligned fall back to demand loads and always prefetch one row)
            const int pf_rows = XT ? (PF_X > 0 ? PF_X + 1 : 0) : (PL::X_TMA ? 1 : PF_X);
            if (pf_rows > 0 && a + pf_rows * AS < p.n_ant)
                prefetch_row<T, false>(x0 + (long long)(a + pf_rows * AS) * p.ant_stride, N, t);
            if (!PL::H_RING && PF_H > 0 && a + PF_H * AS < p.n_ant)
                prefetch_row<T, true>(hw_row + (long long)PF_H * AS * N, N, t);
            const int R = rows_done + a;
            const int st = R % PL::H_STAGES;
            const float2* h_src = PL::H_RING ? (s_hring + st * N) : hw_row;
            bool h_ready = !PL::H_RING;
            row_fft<PL>(v, PL::REG_PF == 1 ? x_next : nullptr, tile, s_tw1, s_tw2, t, team,
                        [&](int sl, int bin, float2 y) {
                            // cpuLS.hpp:187-208: acc += Y * Hconj
                            if constexpr (PL::H_RING) {
                                if (!h_ready) {
                                    mbar_wait(&bar_full[st], (uint32_t)((R / PL::H_STAGES) & 1));
                                    h_ready = true;
                                }
                                acc[sl] = cmac(acc[sl], h_src[PL::hpos(sl, t, bin)], y);
                            } else {
                                const float2 h = __ldg(h_src + PL::hpos(sl, t, bin));
                                if (a_ok) acc[sl] = cmac(acc[sl], h, y);
                            }
                        },
                        tmem,
                        [&]() {
                            if constexpr (XT) {
                                // the tile has been read for the last time in this row: fetch the next row
                                // into it while the last-stage butterflies and the MRC run
                                if (a + 1 < p.n_ant) {
                                    team_sync<PL>(team);
                                    if (t == 0) {
                                        fence_proxy_async();
                                        mbar_expect_tx(&bar_x[team], ROW_BYTES);
                                        bulk_g2s(tile, x0 + (long long)(a + 1) * p.ant_stride, ROW_BYTES, &bar_x[team]);
                                    }
                                }
                            }
                        });
            if constexpr (PL::H_RING) {
                team_sync<PL>(team);
                if (t == 0) mbar_arrive(&bar_empty[st]);
            }
        }
        rows_done += p.n_ant;
        if (AS > 1) {
            // add the antenna slices: slice 0 of every pair sums the others in fixed order
            float2* red = s_tiles;  // [TEAMS][P*T], aliases the tiles (all teams are past their last row)
            __syncthreads();
#pragma unroll
            for (int sl = 0; sl < P; ++sl) red[(team * P + sl) * T + t] = acc[sl];
            __syncthreads();
            if (aj == 0) {
                for (int jj = 1; jj < AS; ++jj) {
#pragma unroll
                    for (int sl = 0; sl < P; ++sl) acc[sl] = cadd(acc[sl], red[((team + jj) * P + sl) * T + t]);
                }
            }
            __syncthreads();
            valid = valid && (aj == 0);
        }

        mrc_finish<PL, false>(p, acc, p.hsqrd + (long long)f * K, f, s, reinterpret_cast<uint8_t*>(my_tiles), valid, t, team);
        team_sync<PL>(team);  // the byte buffer aliases the tile the next item writes
        }  // work items
        if constexpr (PL::TW_TMEM) tmem_free_cols(s_tmem, kTmemCols, (int)(threadIdx.x >> 5));
    }
}

constexpr int kShTmemCols = 128;  // tensor-memory columns per CTA of the shuffle-stage kernels: both twiddle sets of a thread

// ---- row pipeline shared by the two kernels of the shuffle-stage plans -----------------------------------------
// Per-team state of the pipeline in shared memory / tensor memory.
template <class PL>
struct ShRow {
    float2* tile;            // [32][T] dense, columns swizzled (Plan::at)
    uint64_t* bar_x;         // completes on the bytes of the antenna row in flight
    unsigned int* readers;   // warps of the team that have read their stage-2 operands of the current row
    uint32_t tmem;           // this thread's tensor-memory lane: columns [0,64) stage-1, [64,128) stage-2 twiddles
    uint32_t x_phase;
    bool x_tma;
    int t, lane, wt, team, q, k1;
};

// request antenna row `x_row` into the team's tile (one bulk copy; the caller has made sure the tile is free)
template <class PL>
__device__ __forceinline__ void sh_fetch_row(const ShRow<PL>& r, const float2* x_row)
{
    fence_proxy_async();  // the tile's earlier generic-proxy accesses are ordered before the copy
    mbar_expect_tx(r.bar_x, (uint32_t)(PL::N * sizeof(float2)));
    bulk_g2s_hint(r.tile, x_row, (uint32_t)(PL::N * sizeof(float2)), r.bar_x, l2_policy_evict_first());
}

// Everything of a row up to the stage-2 transform: samples out of the tile (or by plain loads when rows are not
// 16-byte aligned), stage 1 with the twiddles from tensor memory, the ONE team barrier of the row, stage-2 operands,
// the request for the next row (x_next, may be nullptr) by whichever warp finishes its reads last, and the
// 32-point stage-2 transform.  `after_barrier()` runs right behind the team barrier: passing it proves that every
// warp of the team is done with the previous row.  On return v[r] holds register r of the stage-2 transform.
template <class PL, class F>
__device__ __forceinline__ void sh_row_front(ShRow<PL>& r, float2 (&v)[32], const float2* x_row, const float2* x_next, F&& after_barrier)
{
    constexpr int T = PL::T, WPT = T / 32;
    if (r.x_tma) {
        mbar_wait(r.bar_x, r.x_phase);
        r.x_phase ^= 1u;
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) v[n1] = r.tile[n1 * T + r.t];  // as the copy laid the row out: linear
        __syncwarp();  // stage 1 writes into columns of this warp's lanes only
    } else {
        row_load<PL>(v, x_row, r.t);
        if (x_next != nullptr) prefetch_row<T, false>(x_next, PL::N, r.t);
    }
    fft_reg<32>(v);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float2 w[8];
        tmem_load8(r.tmem, 16 * c, w);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = 8 * c + i;
            r.tile[PL::at(k, r.t)] = cmul(v[brev<32>(k)], w[i]);
        }
    }
    team_sync<PL>(r.team);
    after_barrier();
    sh_stage2_read<PL>(v, r.tile, r.k1, r.q);
    if (r.x_tma) {
        __syncwarp();
        if (r.lane == 0) {
            if (atomicAdd(r.readers, 1u) == (unsigned)WPT - 1u) {
                *r.readers = 0u;
                if (x_next != nullptr) sh_fetch_row<PL>(r, x_next);
            }
        }
    } else {
        team_sync<PL>(r.team);  // (plain-load fallback: the next row's stage 1 overwrites the tile)
    }
    fft_reg<32>(v);
}

// twiddles of both stages of thread t into its tensor-memory lane (see lsmrc_data_sh)
template <class PL>
__device__ __forceinline__ void sh_fill_tmem(uint32_t tmem, const float2* __restrict__ table, int t, int q)
{
    tmem_fill_stage1<PL>(tmem, table, t);
    const float2* tq = table + PL::TW1 + 2 * q;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        float2 w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = tq[((4 * c + i) / 2) * PL::SH * 2 + ((4 * c + i) & 1)];
        tmem_store4(tmem, 64 + 8 * c, w);
    }
    tmem_store_wait();
}

// ---- data kernel of the shuffle-stage plans (2048 and 4096 points) --------------------------------------------
// Same job as MODE_DATA above (persistent CTAs, one team per (frame, data symbol), antenna loop with the MRC sums in
// registers), restructured around what the shuffle stage frees up:
//  * the tile is needed for ONE exchange only, so it is free as soon as the stage-2 operands have been read -- about
//    40 % into a row.  From there the next antenna row is fetched into it by ONE linear bulk async copy (TMA): the
//    rows of the tile are dense, a thread finds its 32 samples in its own column, and because the column swizzle of
//    stage 1 (Plan::at) only moves data inside aligned groups of 16 lanes, "all samples read" before "stage 1
//    written" is a warp-level dependency, not a team barrier.  The copy is issued by whichever warp of the team
//    finishes its stage-2 reads last (a shared-memory counter), so nobody waits for anybody;
//  * conj(H) of the antenna (slot-major row of hwork, Plan::hpos) is bulk-copied into a per-team buffer right
//    after the one team barrier of the row -- passing it proves that every warp is done with the previous row's
//    values -- and is needed only after the stage-2 transform.
// Neither the samples nor the channel values are waited for on the scoreboard (35 % of all stall samples of the
// round-1 kernels, profiles/r02_before_ncu_c4.txt), and a row costs one team barrier instead of three.
//  * the twiddles of both stages are per-thread constants; they live in tensor memory (see tmem_load8) and cost
//    neither shared-memory wavefronts (a table) nor fp32 instructions (a recurrence).
// Shared memory per CTA: TEAMS x (channel row N + tile N) complex = 64 KB -> 3 CTAs per SM.
// Rows that are not 16-byte aligned (odd prefix lengths) are read with plain 64-bit loads instead of bulk copies.
// One work item of the data kernel: TEAMS consecutive (frame, data symbol) pairs, one per team, all antennas.
// E_CG: sum|H|^2 is read around L1 (the fused kernel: it was written by another CTA of the same launch).
template <class PL, bool E_CG>
__device__ __forceinline__ void sh_data_item(const KernelParams& p, ShRow<PL>& row, float2* hbuf, uint64_t* bar_h, uint32_t& h_phase, int item)
{
    constexpr int N = PL::N, T = PL::T, K = N - 1, SH = PL::SH, TEAMS = PL::TEAMS;
    constexpr uint32_t ROW_BYTES = N * sizeof(float2);
    const int t = row.t, team = row.team, q = row.q;
    const uint32_t tmem = row.tmem;
    const long long n_work = (long long)p.n_frames * p.n_sym_work;
    long long work = (long long)item * TEAMS + team;
    bool valid = work < n_work;
    if (!valid) work = n_work - 1;
    const int f = (int)(work / p.n_sym_work);
    const int s = (int)(work % p.n_sym_work);
    const float2* x0 = p.rx + (long long)f * p.frame_stride + (long long)(p.first_sym + s) * p.sym_stride + p.cp;
    const float2* hw_frame = p.hwork + (long long)f * p.n_ant * N;
    float2 acc[32];
#pragma unroll
    for (int sl = 0; sl < 32; ++sl) acc[sl] = make_float2(0.f, 0.f);

    if (row.x_tma && t == 0) sh_fetch_row<PL>(row, x0);  // (the tile doubled as the previous item's demap byte buffer)
    for (int a = 0; a < p.n_ant; ++a) {
        const float2* x_row = x0 + (long long)a * p.ant_stride;
        float2 v[32];
        sh_row_front<PL>(row, v, x_row, a + 1 < p.n_ant ? x_row + p.ant_stride : nullptr, [&]() {
            // every warp of the team is past the previous antenna: its channel row may be replaced
            if (t == 0) {
                mbar_expect_tx(bar_h, ROW_BYTES);
                bulk_g2s_hint(hbuf, hw_frame + (long long)a * N, ROW_BYTES, bar_h, l2_policy_evict_last());
            }
        });
        // ---- twiddle W_T^(q*k2), radix-SH across the lanes, multiply-accumulate with conj(H)
        constexpr int JB = kShBatch;
        pin_values(v);  // the stage-2 transform stays ahead of the wait: it is the time the channel row has to land
        mbar_wait(bar_h, h_phase);
        h_phase ^= 1u;
#pragma unroll
        for (int c = 0; c < 16 / JB; ++c) {
            float2 tw[2 * JB], h[2 * JB];
            tmem_load8(tmem, 64 + 16 * c, tw);
#pragma unroll
            for (int i = 0; i < 2 * JB; ++i) h[i] = lds_volatile(hbuf + (2 * JB * c + i) * T + t);
            asm volatile("" ::: "memory");
            float2 keep[JB], send[JB], A[JB], B[JB];
#pragma unroll
            for (int i = 0; i < JB; ++i) {
                keep[i] = cmul(v[2 * (JB * c + i)], tw[2 * i]);
                send[i] = cmul(v[2 * (JB * c + i) + 1], tw[2 * i + 1]);
            }
            sh_radix_batch<SH, JB>(keep, send, q, A, B);
            // cpuLS.hpp:187-208: acc += Y * Hconj (both carry the slot's unit factor: it cancels)
#pragma unroll
            for (int i = 0; i < JB; ++i) {
                const int sl = 2 * (JB * c + i);
                acc[sl] = cmac(acc[sl], h[2 * i], A[i]);
                acc[sl + 1] = cmac(acc[sl + 1], h[2 * i + 1], B[i]);
            }
        }
    }
    team_sync<PL>(team);  // every warp is done with the last row before the tile becomes the demap byte buffer
    mrc_finish<PL, false, E_CG>(p, acc, p.hsqrd + (long long)f * K, f, s, reinterpret_cast<uint8_t*>(row.tile), valid, t, team);
    team_sync<PL>(team);  // the byte buffer aliases the tile the next item's first row is copied into
}

// per-CTA set-up shared by the kernels of the shuffle-stage plans: barriers, the reader counters, both twiddle sets into
// this thread's tensor-memory lane (columns [0, 64) the 32 stage-1 factors stage1_sign(t) * W_N^(t*r), columns [64, 128)
// the 32 factors W_T^(q*k2) of its stage-2 registers), and the per-team pipeline state
template <class PL>
__device__ __forceinline__ void sh_setup(const KernelParams& p, ShRow<PL>& row, float2* s_tiles, uint64_t* bar_x, uint64_t* bar_h,
                                         unsigned int* s_readers, uint32_t* s_tmem)
{
    constexpr int T = PL::T, SH = PL::SH, TEAMS = PL::TEAMS, N = PL::N;
    static_assert(PL::THREADS == 128, "one tensor-memory lane per thread: CTAs of exactly four warps");
    const int team = threadIdx.x / T;
    const int t = threadIdx.x % T;
    const int lane = t & 31, wt = t >> 5;
    if (threadIdx.x == 0) {
        for (int i = 0; i < TEAMS; ++i) {
            mbar_init(&bar_x[i], 1);
            if (bar_h) mbar_init(&bar_h[i], 1);
            s_readers[i] = 0u;
        }
        mbar_fence_init();
    }
    // this thread's stage-2 role: row k1 of the tile, lane position q of the shuffle group
    const int q = lane % SH;
    const int k1 = lane / SH + (32 / SH) * wt;
    const uint32_t tmem = tmem_alloc_cols(s_tmem, kShTmemCols, (int)(threadIdx.x >> 5));
    sh_fill_tmem<PL>(tmem, p.twiddles, t, q);
    row.tile = s_tiles + team * N;
    row.bar_x = &bar_x[team];
    row.readers = &s_readers[team];
    row.tmem = tmem;
    row.x_phase = 0;
    row.x_tma = p.x_tma != 0;
    row.t = t, row.lane = lane, row.wt = wt, row.team = team, row.q = q, row.k1 = k1;
}

// draws the next ticket of a persistent kernel (thread 0) and hands it to the whole CTA; -1 when the launch has run out
// of its n_tickets.  The last CTA to find the counter exhausted re-arms it for the next launch (and, with `with_epoch`,
// advances the launch number that the fused kernel's ready flags carry).
template <class TK>
__device__ __forceinline__ TK draw_ticket(const KernelParams& p, TK n_tickets, TK* s_ticket, bool with_epoch)
{
    if (threadIdx.x == 0) {
        const unsigned long long tk = atomicAdd(p.ticket, 1ULL);
        *s_ticket = tk < (unsigned long long)n_tickets ? (TK)tk : -1;
        if (*s_ticket < 0) {
            __threadfence();
            if (atomicAdd(p.ticket + 1, 1ULL) == (unsigned long long)gridDim.x - 1ULL) {
                if (with_epoch) p.ticket[2] = p.ticket[2] + 1ULL;
                p.ticket[0] = 0ULL;
                p.ticket[1] = 0ULL;
            }
        }
    }
    __syncthreads();
    const TK tk = *s_ticket;
    __syncthreads();  // s_ticket is rewritten by thread 0 at the top of the next round
    return tk;
}

template <class PL, int MINB>
__global__ void __launch_bounds__(PL::THREADS, MINB) lsmrc_data_sh(const KernelParams p)
{
    constexpr int N = PL::N, TEAMS = PL::TEAMS;
    static_assert(PL::SH > 1 && PL::ROW == PL::T, "shuffle-stage plans only");
    extern __shared__ __align__(16) float2 smem[];
    float2* s_h = smem;                     // [TEAMS][N]   conj(H) of the current antenna, slot-major
    float2* s_tiles = s_h + TEAMS * N;      // [TEAMS][32][T]
    __shared__ __align__(8) uint64_t bar_x[TEAMS], bar_h[TEAMS];
    __shared__ unsigned int s_readers[TEAMS];  // warps of the team that have read their stage-2 operands of this row
    __shared__ long long s_ticket;
    __shared__ uint32_t s_tmem;
    ShRow<PL> row;
    sh_setup<PL>(p, row, s_tiles, bar_x, bar_h, s_readers, &s_tmem);
    __syncthreads();

    const long long n_work = (long long)p.n_frames * p.n_sym_work;
    const long long n_items = (n_work + TEAMS - 1) / TEAMS;
    uint32_t h_phase = 0;
    for (;;) {
        const long long item = draw_ticket(p, n_items, &s_ticket, false);
        if (item < 0) break;
        sh_data_item<PL, false>(p, row, s_h + row.team * N, &bar_h[row.team], h_phase, (int)item);
    }
    tmem_free_cols(s_tmem, kShTmemCols, (int)(threadIdx.x >> 5));
}

// ---- pilot kernel of the shuffle-stage plans -----------------------------------------------------------------
// Same job as MODE_PILOT above (virtual CTA = (frame, antenna group); teams take the group's antennas round-robin;
// LS estimate, conj, sum_a |H|^2 with the fixed-order cross-team / cross-group sums) on the row pipeline of
// lsmrc_data_sh, so that one pilot row costs what one data row costs -- the generic kernel needed 254 registers
// (8 warps per SM) for the pilot values, reciprocals and energy partials and took twice as long per row.  Here the
// per-bin constant of the LS divide, g = conj(X)/|X|^2 (cpuLS.hpp:240-241 with the reciprocal hoisted), sits in a
// slot-major shared table where the data kernel keeps its channel row, and each thread reads its own 32 entries.
// conj(H) goes to hwork slot-major and factored exactly as the data kernel's outputs are (Plan::unit_mul), so the
// store is coalesced and needs no fix-up; the optional Hconj export in the reference layout is corrected.
// the LS-divide table of a CTA: g = conj(X)/|X|^2 per (slot, thread), slot-major like a channel row; entry of bin 0 is zero
template <class PL>
__device__ __forceinline__ void sh_fill_g(const KernelParams& p, float2* s_g)
{
    constexpr int T = PL::T;
    if (threadIdx.x < T) {
        const int t = threadIdx.x;
#pragma unroll
        for (int sl = 0; sl < 32; ++sl) {
            const int bin = PL::bin_of(sl, t);
            float2 g = make_float2(0.f, 0.f);
            if (bin > 0) {
                const float2 X = p.pilot_bin[bin - 1];
                const float den = 1.0f / (X.x * X.x + X.y * X.y);
                g = make_float2(X.x * den, -X.y * den);
            }
            s_g[sl * T + t] = g;
        }
    }
}

// One virtual CTA of the pilot kernel: antenna group g of frame f (vb = f * n_groups + g), pilot symbol `sym`.
// Returns true in every thread when this call completed the frame's channel state (all of hwork and sum|H|^2 written:
// the only group, or the last group to arrive).
template <class PL>
__device__ __forceinline__ bool sh_pilot_item(const KernelParams& p, ShRow<PL>& row, const float2* s_g, float2* s_tiles, unsigned int* s_last,
                                              int vb, int sym)
{
    constexpr int N = PL::N, T = PL::T, K = N - 1, SH = PL::SH, TEAMS = PL::TEAMS;
    const int t = row.t, team = row.team, q = row.q;
    const uint32_t tmem = row.tmem;
    const int per_iter = p.n_groups * TEAMS;
    const int n_iter = (p.n_ant + per_iter - 1) / per_iter;
    const int f = vb / p.n_groups;
    const int g = vb % p.n_groups;
    const float2* x0 = p.rx + (long long)f * p.frame_stride + (long long)sym * p.sym_stride + p.cp;
    float2* hw_frame = p.hwork + (long long)f * p.n_ant * N;
    float2* hc_frame = p.hconj ? p.hconj + (long long)f * p.n_ant * K : nullptr;
    float e[32];
#pragma unroll
    for (int sl = 0; sl < 32; ++sl) e[sl] = 0.f;
    // antenna of this team in iteration `it`; teams whose share has run out redo the last antenna and drop it
    auto ant_of = [&](int it) { return (it * p.n_groups + g) * TEAMS + team; };
    auto row_of = [&](int it) {
        const int a = ant_of(it);
        return x0 + (long long)(a < p.n_ant ? a : p.n_ant - 1) * p.ant_stride;
    };
    if (row.x_tma && t == 0) sh_fetch_row<PL>(row, row_of(0));
    for (int it = 0; it < n_iter; ++it) {
        const int a_raw = ant_of(it);
        const bool a_ok = a_raw < p.n_ant;
        const int a = a_ok ? a_raw : p.n_ant - 1;
        float2 v[32];
        sh_row_front<PL>(row, v, row_of(it), it + 1 < n_iter ? row_of(it + 1) : nullptr, []() {});
        float2* hw_row = hw_frame + (long long)a * N + t;
        float2* hc_row = hc_frame ? hc_frame + (long long)a * K : nullptr;
        constexpr int JB = kShBatch;
#pragma unroll
        for (int c = 0; c < 16 / JB; ++c) {
            float2 tw[2 * JB], gk[2 * JB];
            tmem_load8(tmem, 64 + 16 * c, tw);
#pragma unroll
            for (int i = 0; i < 2 * JB; ++i) gk[i] = s_g[(2 * JB * c + i) * T + t];
            float2 keep[JB], send[JB], A[JB], B[JB];
#pragma unroll
            for (int i = 0; i < JB; ++i) {
                keep[i] = cmul(v[2 * (JB * c + i)], tw[2 * i]);
                send[i] = cmul(v[2 * (JB * c + i) + 1], tw[2 * i + 1]);
            }
            sh_radix_batch<SH, JB>(keep, send, q, A, B);
#pragma unroll
            for (int i = 0; i < 2 * JB; ++i) {
                const int sl = 2 * JB * c + i;
                const float2 z = (i & 1) ? B[i / 2] : A[i / 2];
                // LS estimate H = Z / X (cpuLS.hpp:233-244) as Z * conj(X)/|X|^2, then conj (:303-307); z, and so
                // hc, carry the slot's unit factor, the energy does not care
                const float re = z.x * gk[i].x - z.y * gk[i].y;
                const float im = z.x * gk[i].y + z.y * gk[i].x;
                if (a_ok) {
                    const float2 hc = make_float2(re, -im);
                    hw_row[sl * T] = hc;
                    if (hc_row) {
                        const int bin = PL::bin_of(sl, t);
                        if (bin > 0) hc_row[bin - 1] = PL::refix(sl, t, hc);
                    }
                    e[sl] += re * re + im * im;  // cpuLS.hpp:211-228 (the entry of bin 0 is zero)
                }
            }
        }
    }
    // deterministic cross-team sum of the energy partials, then cross-group by the last CTA of the frame
    __syncthreads();
    float* s_e = reinterpret_cast<float*>(s_tiles);  // [TEAMS][N] indexed by bin; aliases the tiles (no copy is in flight)
#pragma unroll
    for (int sl = 0; sl < 32; ++sl) s_e[team * N + PL::bin_of(sl, t)] = e[sl];
    __syncthreads();
    for (int bin = 1 + (int)threadIdx.x; bin < N; bin += PL::THREADS) {
        float acc = s_e[bin];
#pragma unroll
        for (int tm = 1; tm < TEAMS; ++tm) acc += s_e[tm * N + bin];
        float* dst = (p.n_groups == 1) ? (p.hsqrd + (long long)f * K - 1) : (p.epart + ((long long)f * p.n_groups + g) * N);
        dst[bin] = acc;
    }
    bool completed = p.n_groups == 1;
    if (p.n_groups > 1) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned int prev = atomicAdd(p.counters + f, 1u);
            *s_last = (prev == (unsigned)p.n_groups - 1u);
            if (*s_last) p.counters[f] = 0u;  // self-reset for the next launch
        }
        __syncthreads();
        if (*s_last) {
            __threadfence();
            const float* ep = p.epart + (long long)f * p.n_groups * N;
            for (int bin = 1 + (int)threadIdx.x; bin < N; bin += PL::THREADS) {
                float acc = __ldcg(ep + bin);
                for (int gg = 1; gg < p.n_groups; ++gg) acc += __ldcg(ep + (long long)gg * N + bin);
                p.hsqrd[(long long)f * K + bin - 1] = acc;
            }
            completed = true;
        }
    }
    __syncthreads();  // the partial-energy buffer aliases the tiles the next virtual CTA copies into
    return completed;
}

template <class PL, int MINB>
__global__ void __launch_bounds__(PL::THREADS, MINB) lsmrc_pilot_sh(const KernelParams p)
{
    constexpr int N = PL::N, TEAMS = PL::TEAMS;
    static_assert(PL::SH > 1 && PL::ROW == PL::T && PL::THREADS == 128, "shuffle-stage plans only");
    extern __shared__ __align__(16) float2 smem[];
    float2* s_g = smem;                 // [32][T] conj(X)/|X|^2 of (slot, thread)
    float2* s_tiles = s_g + N;          // [TEAMS][32][T]
    __shared__ __align__(8) uint64_t bar_x[TEAMS];
    __shared__ unsigned int s_readers[TEAMS];
    __shared__ uint32_t s_tmem;
    __shared__ unsigned int s_last;
    ShRow<PL> row;
    sh_setup<PL>(p, row, s_tiles, bar_x, nullptr, s_readers, &s_tmem);
    sh_fill_g<PL>(p, s_g);
    __syncthreads();
    const int n_virtual = p.n_frames * p.n_groups;
    for (int vb = blockIdx.x; vb < n_virtual; vb += gridDim.x) sh_pilot_item<PL>(p, row, s_g, s_tiles, &s_last, vb, p.first_sym);
    tmem_free_cols(s_tmem, kShTmemCols, (int)(threadIdx.x >> 5));
}

// ---- both in one launch: pilot and data items on one ticket counter -------------------------------------------------
// The persistent CTAs draw BOTH kinds of item from one counter: first the pilot items of every frame (frame-major), then the
// data items.  Compared with the kernel pair there is no drain / launch / ramp between the two phases -- CTAs that run out of
// pilot items start on the data items of the first frames while the last pilot items are still running.  A data item waits
// (one thread, acquire loads) until the pilot of its frame(s) has signalled completion -- ready[f] = number of this launch,
// written with release semantics by the CTA that completed frame f.  Every pilot item has a smaller ticket than every data
// item, i.e. is running or done on a resident CTA, and pilot items never wait: the kernel cannot deadlock whatever the grid
// size.  The launch number lives on the device next to the counter (ticket[2], advanced by the last CTA to leave), so a
// launch carries no host-side state.  Channel rows and sum|H|^2 are read around L1 (bulk copies, ld.cg): other CTAs of the
// same launch write them.
// Measured and rejected: INTERLEAVING pilot items of later frames with the data items of earlier ones (the pilot work is
// DRAM-bound, the data work is not, so they looked like they would overlap).  The data items are latency-bound with one row
// of prefetch; the extra DRAM traffic next to them raises their bulk-copy waits more than the overlap saves (c4, 192 frames:
// 5.03 ms pilots first, 5.35-5.8 ms interleaved with 50 / 32 / 16 / 8 frames of lead; the kernel pair 5.19 ms).
__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p)
{
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned int* p, unsigned int v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

template <class PL, int MINB>
__global__ void __launch_bounds__(PL::THREADS, MINB) lsmrc_frames_sh(const KernelParams p)
{
    constexpr int N = PL::N, TEAMS = PL::TEAMS;
    static_assert(PL::SH > 1 && PL::ROW == PL::T && PL::THREADS == 128, "shuffle-stage plans only");
    extern __shared__ __align__(16) float2 smem[];
    float2* s_h = smem;                     // data items: [TEAMS][N] conj(H) of the current antenna; pilot items: [N] LS-divide table
    float2* s_tiles = s_h + TEAMS * N;      // [TEAMS][32][T]
    __shared__ __align__(8) uint64_t bar_x[TEAMS], bar_h[TEAMS];
    __shared__ unsigned int s_readers[TEAMS];
    __shared__ long long s_ticket;
    __shared__ uint32_t s_tmem;
    __shared__ unsigned int s_last;
    ShRow<PL> row;
    sh_setup<PL>(p, row, s_tiles, bar_x, bar_h, s_readers, &s_tmem);
    const unsigned int epoch = (unsigned int)__ldcg(p.ticket + 2) + 1u;  // (every CTA reads it before the last one to leave advances it)
    __syncthreads();

    const long long np = (long long)p.n_frames * p.n_groups;  // pilot items, frame-major
    const long long n_work = (long long)p.n_frames * p.n_sym_work;
    const long long nd = (n_work + TEAMS - 1) / TEAMS;         // data items
    const long long n_tickets = np + nd;
    bool g_valid = false;  // the LS-divide table sits where data items keep their channel rows
    uint32_t h_phase = 0;
    for (;;) {
        const long long tk = draw_ticket(p, n_tickets, &s_ticket, true);
        if (tk < 0) break;
        const long long pilot = tk < np ? tk : -1, data = tk - np;
        if (pilot >= 0) {
            if (!g_valid) {
                sh_fill_g<PL>(p, s_h);
                g_valid = true;
                __syncthreads();
            }
            const bool completed = sh_pilot_item<PL>(p, row, s_h, s_tiles, &s_last, (int)pilot, 0);
            if (completed) {
                __threadfence();   // every thread's channel rows / energy sums, then the flag
                __syncthreads();
                if (threadIdx.x == 0) {
                    fence_proxy_async_all();
                    st_release_gpu(p.ready + pilot / p.n_groups, epoch);
                }
            }
        } else {
            // the frames of this item's (frame, symbol) pairs: first and last differ at most by one
            const long long w0 = data * TEAMS, w1 = (w0 + TEAMS - 1 < n_work ? w0 + TEAMS - 1 : n_work - 1);
            const int f0 = (int)(w0 / p.n_sym_work), f1 = (int)(w1 / p.n_sym_work);
            if (threadIdx.x == 0) {
                while (ld_acquire_gpu(p.ready + f0) != epoch) __nanosleep(200);
                while (ld_acquire_gpu(p.ready + f1) != epoch) __nanosleep(200);
            }
            __syncthreads();
            fence_proxy_async_all();  // the channel rows are fetched by bulk copies (async proxy)
            g_valid = false;
            sh_data_item<PL, true>(p, row, s_h + row.team * N, &bar_h[row.team], h_phase, (int)data);
            __syncthreads();  // (a pilot item may follow and rebuild its table over the channel rows of slower teams)
        }
    }
    tmem_free_cols(s_tmem, kShTmemCols, (int)(threadIdx.x >> 5));
}

// ---- stand-alone per-step kernels: the individually callable steps of gpuLS.cuh:87-99 -----------
// (the fused kernels above never use them; they exist so that callers of the reference's
// wrapper methods get the same intermediate tensors)

// gpuLS.cu:143-156 dropPrefix: out[r][n] = in[r][n + cp]
__global__ void k_drop_prefix(float2* __restrict__ out, const float2* __restrict__ in, long long rows, int n, int cp)
{
    const long long total = rows * n;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / n;
        const int c = (int)(i - r * n);
        out[i] = in[r * (n + cp) + cp + c];
    }
}

// Receive front end, sample format.  The radio's wire format is interleaved int16 I/Q: rx_and_corr.cpp:283 asks UHD for cpu
// format "fc32" over wire format "sc16", i.e. UHD converts on the host (fc32 = sc16 * scale, scale = 1/32767 by default) and
// the reference ships 8 bytes per sample to the GPU.  Here the wire format crosses PCIe (half the bytes) and is converted on
// the device, dropping `skip` leading samples of every row (the cyclic prefix) on the way:
// out[r][n] = float(in[r][skip + n]) * scale -- int16 -> float is exact and the product is one rounding, so the result is
// bit-identical to the host conversion.  VEC2: two samples per thread (n_in, skip, n_out even; 8-byte loads, 16-byte stores).
template <bool VEC2>
__global__ void k_sc16_to_fc32(float2* __restrict__ out, const short2* __restrict__ in, long long rows, int n_in, int skip, int n_out,
                               float scale)
{
    constexpr int V = VEC2 ? 2 : 1;
    const int per_row = n_out / V;
    const long long total = rows * per_row;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / per_row;
        const int c = (int)(i - r * per_row) * V;
        if constexpr (VEC2) {
            const int2 w = *reinterpret_cast<const int2*>(in + r * n_in + skip + c);
            const short2 a = *reinterpret_cast<const short2*>(&w.x), b = *reinterpret_cast<const short2*>(&w.y);
            float4 o;
            o.x = __int2float_rn(a.x) * scale, o.y = __int2float_rn(a.y) * scale;
            o.z = __int2float_rn(b.x) * scale, o.w = __int2float_rn(b.y) * scale;
            *reinterpret_cast<float4*>(out + r * n_out + c) = o;
        } else {
            const short2 a = in[r * n_in + skip + c];
            out[r * n_out + c] = make_float2(__int2float_rn(a.x) * scale, __int2float_rn(a.y) * scale);
        }
    }
}

// gpuLS.cu:158-182 findHs: hconj[a][k] = conj(yfft[a][k+1] / x[k])   (x: K entries, bin order)
__global__ void k_find_hs(const float2* __restrict__ yfft, float2* __restrict__ hconj, const float2* __restrict__ x,
                          int rows, int n, int x_row_stride)
{
    const int K = n - 1;
    const long long total = (long long)rows * K;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(i / K), k = (int)(i - (long long)a * K);
        const float2 z = yfft[(long long)a * n + k + 1];
        const float2 X = x[(long long)a * x_row_stride + k];
        const float den = X.x * X.x + X.y * X.y;
        hconj[i] = make_float2((z.x * X.x + z.y * X.y) / den, -((z.y * X.x - z.x * X.y) / den));
    }
}

// gpuLS.cu:185-209 findDistSqrd: hsqrd[k] = sum_a |h[a][k]|^2  (sequential over a: the CPU order)
__global__ void k_find_hsqrd(const float2* __restrict__ h, float* __restrict__ hsqrd, int rows, int K)
{
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
        float acc = 0.f;
        for (int a = 0; a < rows; ++a) {
            const float2 v = h[(long long)a * K + k];
            acc += v.x * v.x + v.y * v.y;
        }
        hsqrd[k] = acc;
    }
}

// gpuLS.cu:212-233 multiplyWithChannelConj: yf[s][a][k] = yfft[s][a][k+1] * hconj[a][k]
__global__ void k_mult_conj(const float2* __restrict__ yfft, const float2* __restrict__ hconj, float2* __restrict__ yf,
                            int syms, int rows, int n)
{
    const int K = n - 1;
    const long long per_sym = (long long)rows * K, total = per_sym * syms;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long sy = i / per_sym, r = i - sy * per_sym;
        const int a = (int)(r / K), k = (int)(r - (long long)a * K);
        yf[i] = cmul(yfft[(sy * rows + a) * n + k + 1], hconj[r]);
    }
}

// gpuLS.cu:236-259 combineForMRC: out[s][k] = (sum_a yf[s][a][k]) / hsqrd[k]   (out must not alias yf)
__global__ void k_combine(const float2* __restrict__ yf, const float* __restrict__ hsqrd, float2* __restrict__ out, int syms,
                          int rows, int K)
{
    const long long total = (long long)syms * K;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long sy = i / K;
        const int k = (int)(i - sy * K);
        float2 acc = make_float2(0.f, 0.f);
        for (int a = 0; a < rows; ++a) acc = cadd(acc, yf[(sy * rows + a) * K + k]);
        const float e = hsqrd[k];
        out[i] = make_float2(acc.x / e, acc.y / e);
    }
}

// gpuLS.cu:109-125 shiftOneRow: out[r][i] = in[r][(i + (K-1)/2) mod K]   (out must not alias in)
__global__ void k_shift_rows(const float2* __restrict__ in, float2* __restrict__ out, long long rows, int K)
{
    const long long total = rows * K;
    const int sh = (K - 1) / 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / K;
        const int c = (int)(i - r * K);
        int src = c + sh;
        if (src >= K) src -= K;
        out[i] = in[r * K + src];
    }
}

// ---- receive front end before the hot path (SURVEY 8f rank 1; rx_and_corr.cpp:332-393) ----------------

// PN-sequence frame sync, rx_and_corr.cpp:335-360: metric[ch][i] = |sum_j pn[j]*buf[ch][i+j]| / L for every
// channel and offset at once (the reference scans them one by one on the CPU and stops at the first hit).
// The first hit in the reference's scan order (channel-major, offset ascending) is the minimum of
// key = (ch*samps + i) << 32 | float_bits(metric) over all positions with metric >= thres.
// Products and sums are rounded separately in tap order, exactly as the (un-contracted) CPU loop does.
constexpr int kSyncThreads = 256;
__global__ void __launch_bounds__(kSyncThreads) k_sync_correlate(const float2* __restrict__ buf, int samps,
                                                                  const float2* __restrict__ pn, int L, float thres,
                                                                  unsigned long long* __restrict__ first_hit,
                                                                  float* __restrict__ metric_all)
{
    extern __shared__ float2 s_sync[];  // [L] pn, then [kSyncThreads + L - 1] samples
    float2* s_pn = s_sync;
    float2* s_x = s_sync + L;
    const int ch = blockIdx.y;
    const int i0 = blockIdx.x * kSyncThreads;
    const int n_off = samps - L + 1;
    const float2* x = buf + (long long)ch * samps;
    for (int j = threadIdx.x; j < L; j += kSyncThreads) s_pn[j] = pn[j];
    for (int j = threadIdx.x; j < kSyncThreads + L - 1; j += kSyncThreads)
        s_x[j] = (i0 + j < samps) ? x[i0 + j] : make_float2(0.f, 0.f);
    __syncthreads();
    const int i = i0 + threadIdx.x;
    if (i >= n_off) return;
    float re = 0.f, im = 0.f;
    const float2* w = s_x + threadIdx.x;
    for (int j = 0; j < L; ++j) {
        const float2 p = s_pn[j], v = w[j];
        re = __fadd_rn(re, __fsub_rn(__fmul_rn(p.x, v.x), __fmul_rn(p.y, v.y)));
        im = __fadd_rn(im, __fadd_rn(__fmul_rn(p.x, v.y), __fmul_rn(p.y, v.x)));
    }
    const float m = __fdiv_rn(__fsqrt_rn(__fadd_rn(__fmul_rn(re, re), __fmul_rn(im, im))), (float)L);
    if (metric_all) metric_all[(long long)ch * samps + i] = m;
    if (m >= thres) {
        const unsigned long long key = ((unsigned long long)((long long)ch * samps + i) << 32) | (unsigned long long)__float_as_uint(m);
        atomicMin(first_hit, key);
    }
}

// Frame stitching + slot gather, rx_and_corr.cpp:372-393 and :64-87 in one pass: the frame starts right
// after the PN sequence at buf1[ch][off+L] and wraps into buf2; rx[s][a][n] = frame[a][s*(N+C) + n] with the
// cyclic prefix left in (the fused kernels strip it).
__global__ void k_sync_assemble(const float2* __restrict__ buf1, const float2* __restrict__ buf2, int samps, int off,
                                int L, float2* __restrict__ rx, int S, int A, int row)
{
    const long long total = (long long)S * A * row;
    const int n_first = samps - off - L;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i % row);
        const long long sa = i / row;
        const int a = (int)(sa % A);
        const int s = (int)(sa / A);
        const int m = s * row + n;
        rx[i] = (m < n_first) ? buf1[(long long)a * samps + off + L + m] : buf2[(long long)a * samps + (m - n_first)];
    }
}

// ---- soft-output helpers on the receiver's outputs (SURVEY 8f rank 2; nothing in the reference) ------------

// nearest constellation level of one axis, same comparisons as demap_symbol()
template <int B>
__device__ __forceinline__ float slice_axis(float u)
{
    const float au = fabsf(u);
    float lev;
    if (B == 2) {
        lev = (float)0.7071067811865476;
    } else if (B == 4) {
        const float a = (float)0.31622776601683794;
        lev = (au > (float)0.6324555320336759) ? 3.0f * a : a;
    } else {
        const float a = (float)0.1543033499620919;
        const float t4 = (float)0.6172133998483676, t2 = (float)0.3086066999241838;
        const bool outer = au > t4, far = fabsf(__fsub_rn(au, t4)) > t2;
        lev = outer ? (far ? 7.0f * a : 5.0f * a) : (far ? a : 3.0f * a);
    }
    return u < 0.0f ? -lev : lev;
}

// Decision-directed noise estimate, step 1: CTA (row) sums  E[bin(i)] * |y_i - slice(y_i)|^2  over the K
// symbols of one combined row [F*(S-1)][K] (ascending frequency) into part[row].  Fixed reduction
// order (per-thread strided sums, warp shuffles, then warps in order): deterministic.
template <int B>
__device__ __forceinline__ void noise_row(const float2* __restrict__ y, const float* __restrict__ e_bin, int K, float* part_out)
{
    float acc = 0.f;
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        const float2 v = y[i];
        const float dr = __fsub_rn(v.x, slice_axis<B>(v.x)), di = __fsub_rn(v.y, slice_axis<B>(v.y));
        int k = i + (K - 1) / 2;
        if (k >= K) k -= K;
        acc += e_bin[k] * (dr * dr + di * di);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    __shared__ float s_w[32];
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) t += s_w[w];
        *part_out = t;
    }
}

__global__ void k_noise_rows(const float2* __restrict__ combined, const float* __restrict__ hsqrd, int K, int rows_per_frame,
                             int qam_bits, float* __restrict__ part)
{
    const long long row = blockIdx.x;
    const int f = (int)(row / rows_per_frame);
    const float2* y = combined + row * K;
    const float* e = hsqrd + (long long)f * K;
    if (qam_bits == 2) noise_row<2>(y, e, K, part + row);
    else if (qam_bits == 4) noise_row<4>(y, e, K, part + row);
    else noise_row<6>(y, e, K, part + row);
}

// step 2: noise_var[f] = sum_s part[f][s] / (rows_per_frame * K), one warp per frame, fixed order
__global__ void k_noise_frames(const float* __restrict__ part, int rows_per_frame, int K, int n_frames, float* __restrict__ noise_var)
{
    const int f = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (f >= n_frames) return;
    const int lane = threadIdx.x & 31;
    float acc = 0.f;
    for (int s = lane; s < rows_per_frame; s += 32) acc += part[(long long)f * rows_per_frame + s];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) noise_var[f] = acc / ((float)rows_per_frame * (float)K);
}

// LLRs of combined symbols with a per-frame noise variance: llr [F][S-1][K][B], same formula as the
// data kernel's soft epilogue (soft_symbol) with rho = E[bin(i)] / noise_var[f]
template <int B>
__global__ void k_llr_rows(const float2* __restrict__ combined, const float* __restrict__ hsqrd, const float* __restrict__ noise_var,
                           int K, int rows_per_frame, long long n_sym, float* __restrict__ llr)
{
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n_sym; idx += (long long)gridDim.x * blockDim.x) {
        const long long row = idx / K;
        const int i = (int)(idx - row * K);
        const int f = (int)(row / rows_per_frame);
        int k = i + (K - 1) / 2;
        if (k >= K) k -= K;
        const float2 v = combined[idx];
        const float rho = __fmul_rn(hsqrd[(long long)f * K + k], __frcp_rn(noise_var[f]));
        float l[B];
        soft_symbol<B>(v.x, v.y, rho, l);
#pragma unroll
        for (int q = 0; q < B; ++q) llr[idx * B + q] = l[q];
    }
}

// ---- multi-user zero forcing (SURVEY 8f rank 4; cpuLS.hpp:400-463, uncalled in the reference) ---------------
// createZeroForcingMatrix: per subcarrier k, with Xk = X[:, :, k] (U users x A antennas),
//   Hk = Xk^H * inv(Xk * Xk^H + lambda*I)   (A x U, column-major, ld = A)  ->  Hzf[k][u][a].
// A CTA takes KT (<= kZfKT, chosen by the launcher so that the tile fits shared memory) consecutive subcarriers so that
// the gather from X [U][A][K] reads KT contiguous samples per (user, antenna); Gram matrix, inverse (Gauss-Jordan with
// partial pivoting, one thread per subcarrier -- U is a handful) and the A x U product all run out of shared memory.
// Singular subcarriers (a pivot below 1e-6 of the largest Gram entry) yield a zero block and are counted in *n_singular.
// blockIdx.y is the frame: X and Hzf of frame f start at f * x_frame_stride / f * hzf_frame_stride; user u's rows of X
// at u * x_user_stride.  Per subcarrier the result depends on neither KT nor the frame batch.
// With X = conj(H) (H the A x U channel of subcarrier k), Hzf[k][u][a] = conj(W_k[u][a]) for the linear detector
// W_k = inv(H^H H + lambda*I) H^H: ZF at lambda = 0, MMSE at lambda = noise variance (DESIGN.md 8e).
// ginv_diag (may be nullptr) [frame][U][K]: the real diagonal of M_k = inv(G_k), 0 on a singular subcarrier -- what the
// soft output of the multi-user path needs (DESIGN.md 8f).
constexpr int kZfKT = 8;
constexpr int kZfMaxUsers = 16;

__global__ void k_zf_create(const float2* __restrict__ X, float2* __restrict__ Hzf, int A, int K, int U, int KT, float lambda,
                            long long x_frame_stride, long long x_user_stride, long long hzf_frame_stride, int* n_singular,
                            float* __restrict__ ginv_diag)
{
    extern __shared__ __align__(16) float2 zsm[];
    float2* s_x = zsm;                      // [KT][A][U]  (users x antennas, column-major per subcarrier)
    float2* s_g = s_x + (size_t)KT * A * U;  // [KT][U][2U] augmented rows for the inverse
    __shared__ int s_ok[kZfKT];
    X += (long long)blockIdx.y * x_frame_stride;
    Hzf += (long long)blockIdx.y * hzf_frame_stride;
    const int k0 = blockIdx.x * KT;
    const int nk = min(KT, K - k0);
    for (int idx = threadIdx.x; idx < U * A * KT; idx += blockDim.x) {
        const int kt = idx % KT, ua = idx / KT;  // ua = u*A + a, kt fastest: contiguous in X
        const int u = ua / A, a = ua - u * A;
        s_x[((size_t)kt * A + a) * U + u] = (kt < nk) ? X[(long long)u * x_user_stride + (long long)a * K + k0 + kt] : make_float2(0.f, 0.f);
    }
    __syncthreads();
    // Gram matrix G[u][v] = sum_a x[u,a] * conj(x[v,a]) (+ lambda on the diagonal) into the left half of the augmented
    // rows, identity right
    for (int idx = threadIdx.x; idx < KT * U * U; idx += blockDim.x) {
        const int kt = idx / (U * U), r = idx % (U * U), u = r / U, v = r % U;
        const float2* xk = s_x + (size_t)kt * A * U;
        float2 acc = make_float2(0.f, 0.f);
        for (int a = 0; a < A; ++a) {
            const float2 p = xk[a * U + u], q = xk[a * U + v];
            acc.x += p.x * q.x + p.y * q.y;
            acc.y += p.y * q.x - p.x * q.y;
        }
        if (u == v) acc.x += lambda;  // (a diagonal sum is >= +0: adding lambda = 0 leaves it bit for bit)
        float2* row = s_g + ((size_t)kt * U + u) * 2 * U;
        row[v] = acc;
        row[U + v] = make_float2(u == v ? 1.f : 0.f, 0.f);
    }
    __syncthreads();
    if (threadIdx.x < KT) {
        const int kt = threadIdx.x;
        float2* w = s_g + (size_t)kt * U * 2 * U;
        bool ok = kt < nk;
        // a pivot below 1e-6 of the largest Gram entry is rounding noise in fp32: the subcarrier is singular
        float gmax = 0.f;
        for (int i = 0; i < U; ++i)
            for (int j = 0; j < U; ++j) gmax = fmaxf(gmax, fabsf(w[i * 2 * U + j].x) + fabsf(w[i * 2 * U + j].y));
        const float tiny = 1e-6f * gmax;
        for (int c = 0; c < U && ok; ++c) {
            int piv = c;
            float best = -1.f;
            for (int i = c; i < U; ++i) {
                const float m = fabsf(w[i * 2 * U + c].x) + fabsf(w[i * 2 * U + c].y);
                if (m > best) {
                    best = m;
                    piv = i;
                }
            }
            if (!(best > tiny)) {
                ok = false;
                break;
            }
            if (piv != c)
                for (int j = 0; j < 2 * U; ++j) {
                    const float2 tmp = w[c * 2 * U + j];
                    w[c * 2 * U + j] = w[piv * 2 * U + j];
                    w[piv * 2 * U + j] = tmp;
                }
            const float2 pv = w[c * 2 * U + c];
            const float den = 1.0f / (pv.x * pv.x + pv.y * pv.y);
            const float2 pinv = make_float2(pv.x * den, -pv.y * den);
            for (int j = 0; j < 2 * U; ++j) {
                const float2 e = w[c * 2 * U + j];
                w[c * 2 * U + j] = make_float2(e.x * pinv.x - e.y * pinv.y, e.x * pinv.y + e.y * pinv.x);
            }
            for (int i = 0; i < U; ++i) {
                if (i == c) continue;
                const float2 f = w[i * 2 * U + c];
                for (int j = 0; j < 2 * U; ++j) {
                    const float2 e = w[c * 2 * U + j];
                    w[i * 2 * U + j].x -= f.x * e.x - f.y * e.y;
                    w[i * 2 * U + j].y -= f.x * e.y + f.y * e.x;
                }
            }
        }
        s_ok[kt] = ok ? 1 : 0;
        if (kt < nk && !ok && n_singular) atomicAdd(n_singular, 1);
    }
    __syncthreads();
    // Hk[a][u] = sum_v conj(x[v,a]) * Ginv[v][u]; a fastest so the store is coalesced
    for (int idx = threadIdx.x; idx < KT * U * A; idx += blockDim.x) {
        const int kt = idx / (U * A), r = idx % (U * A), u = r / A, a = r % A;
        if (kt >= nk) continue;
        const float2* xk = s_x + (size_t)kt * A * U;
        const float2* gi = s_g + (size_t)kt * U * 2 * U + U;  // right half: row v, column u at gi[v*2U + u]
        float2 acc = make_float2(0.f, 0.f);
        if (s_ok[kt]) {
            for (int v = 0; v < U; ++v) {
                const float2 p = xk[a * U + v], q = gi[v * 2 * U + u];
                acc.x += p.x * q.x + p.y * q.y;
                acc.y += p.x * q.y - p.y * q.x;
            }
        }
        Hzf[(size_t)(k0 + kt) * A * U + (size_t)u * A + a] = acc;
    }
    // the row swaps are row operations of [G | I] as well: the right half is inv(G) itself, no permutation to undo.
    // (A loop of its own after the product, where few registers are live: the kernel keeps its register count.)
    if (ginv_diag != nullptr) {
        float* gd = ginv_diag + (long long)blockIdx.y * U * K + k0;
        for (int idx = threadIdx.x; idx < U * nk; idx += blockDim.x) {
            const int u = idx / nk, kt = idx - u * nk;  // kt fastest: contiguous in ginv_diag
            gd[(long long)u * K + kt] = s_ok[kt] ? s_g[((size_t)kt * U + u) * 2 * U + U + u].x : 0.f;
        }
    }
}

// multiplyWithChannelInv: HX[a][k] = sum_u Hk[a + A*u] * Xd[u][k]
__global__ void k_zf_apply(const float2* __restrict__ Hzf, const float2* __restrict__ Xd, float2* __restrict__ HX, int A, int K, int U)
{
    const long long n = (long long)A * K;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(idx / A), a = (int)(idx - (long long)k * A);  // a fastest: coalesced Hzf reads
        float2 acc = make_float2(0.f, 0.f);
        for (int u = 0; u < U; ++u) {
            const float2 h = Hzf[(size_t)k * A * U + (size_t)u * A + a], x = Xd[(size_t)u * K + k];
            acc.x += h.x * x.x - h.y * x.y;
            acc.y += h.x * x.y + h.y * x.x;
        }
        HX[(size_t)a * K + k] = acc;
    }
}

// ---- multi-user detection (DESIGN.md 8e) ----------------------------------------------------------------------
// Frame [S][A][N+C] with U users: symbol u < U is user u's pilot (the others silent), symbols U..S-1 carry all users.
// Per-user conj(H) comes from the pilot kernel run once per pilot symbol, the detector W_k (U x A per subcarrier) from
// k_zf_create as conj(Hzf).  The data kernel never stores the FFT output: per (frame, data symbol, group of UG users) a
// team transforms each antenna row and accumulates x^[u][k] += Wd[u][a][slot] * y'[slot] in registers.

// Wd [F][UP][A][N]: W_k[u][a] in the plan's slot layout (Plan::hpos), times conj of the slot's unit factor (the sink
// of row_fft sees y' = u * Y on the shuffle-stage plans, so Wd * y' = W * Y).  Users U..UP-1 (padding of the last
// group) and bin 0 are zero.  Hzf [F][K][U][A] = conj(W).
// BIN_ORDER: plain bin order instead of the slot layout, no unit factor -- the downlink precoder (DESIGN.md 8g) feeds W
// to the FFT's input, which is natural order on every plan.  (On plans without a shuffle stage the two layouts are the
// same, so those only need the default instantiation.)
template <class PL, bool BIN_ORDER = false>
__global__ void k_mu_weights(const float2* __restrict__ hzf, float2* __restrict__ wd, int A, int U, int UP, long long rows)
{
    constexpr int N = PL::N, T = PL::T, K = N - 1;
    constexpr bool SLOTS = PL::SH > 1 && !BIN_ORDER;
    const long long n = rows * N;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
        const int pos = (int)(idx % N);
        const long long row = idx / N;  // (f * UP + u) * A + a
        const int a = (int)(row % A);
        const int u = (int)((row / A) % UP);
        const long long f = row / ((long long)A * UP);
        const int sl = pos / T, t = pos % T;
        const int bin = SLOTS ? PL::bin_of(sl, t) : pos;
        float2 w = make_float2(0.f, 0.f);
        if (bin > 0 && u < U) {
            const float2 c = hzf[((f * K + (bin - 1)) * U + u) * A + a];
            w = make_float2(c.x, -c.y);
            if constexpr (SLOTS) w = PL::unfix(sl, t, w);
        }
        wd[idx] = w;
    }
}

// Soft output of the linear detector (DESIGN.md 8f): per (frame, user, subcarrier) from d = [inv(G_k)]_uu (k_zf_create's
// ginv_diag, [F][U][K] bin order k = bin - 1) the pair (rho, scale) the data kernel's soft epilogue needs:
//   ZF   (mmse = 0):  rho = 1 / (sigma2 d),              scale = 1
//   MMSE (mmse = 1):  rho = 1 / (lambda d) - 1 (>= 0),   scale = 1 / beta,  beta = 1 - lambda d = [W H]_uu
// (rho of MMSE straight from lambda d: 1 - beta cancels in fp32 at high SNR).  d = 0 (singular subcarrier) or rho <= 0
// give (0, 0): every LLR of that subcarrier is 0.  sinr (may be nullptr) [F][U][K] gets rho in ascending frequency.
__global__ void k_mu_soft_scale(const float* __restrict__ ginv_diag, float2* __restrict__ tab, float* __restrict__ sinr, long long n,
                                int K, int mmse, float lambda, float sigma2)
{
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
        const float d = ginv_diag[idx];
        float rho = 0.f, scale = 0.f;
        if (d > 0.f) {
            if (mmse) {
                const float ld = lambda * d;
                rho = 1.0f / ld - 1.0f;
                if (rho > 0.f) scale = 1.0f / (1.0f - ld);
                else rho = 0.f;
            } else {
                rho = 1.0f / (sigma2 * d);
                scale = 1.0f;
            }
        }
        tab[idx] = make_float2(rho, scale);
        if (sinr != nullptr) {
            const long long fu = idx / K;
            const int bin = (int)(idx - fu * K) + 1, half = (K + 1) / 2;
            sinr[fu * K + (bin < half ? bin - 1 + half : bin - half)] = rho;
        }
    }
}

// Comb pilots (DESIGN.md 8h): symbol 0 carries user u's pilot on the ascending-frequency indices i = u (mod U) only.
// From the LS estimate of that one symbol, ls [rows = F*A][K] = conj(Z0 / X) in bin order (the pilot kernel's export),
// every user's conj(H) on every subcarrier, out [U][rows][K] (user_stride between users), bin order:
//   own pilot (i = u mod U)               ls[i], copied;
//   between u's pilots p0 < i < p1        ls[p0] + w (ls[p1] - ls[p0]),  w = (phi(i) - phi(p0)) / (phi(p1) - phi(p0));
//   beyond u's outermost pilot            the nearest pilot's ls, held.
// phi(i) = i - N/2 for i < N/2, i - N/2 + 1 above: the signed frequency, without DC.  Bin-order index k holds ascending
// i = (k + N/2) mod K.  A CTA takes one (frame, antenna) row at a time, staged in shared memory (K float2); threads run
// over the output index k, so each user's output row is one coalesced store.
__global__ void k_mu_comb_interp(const float2* __restrict__ ls, float2* __restrict__ out, int N, int U, long long rows,
                                 long long user_stride)
{
    extern __shared__ float2 s_row[];
    const int K = N - 1, half = N / 2;
    auto phi = [&](int i) { return i < half ? i - half : i - half + 1; };
    auto bin = [&](int i) { return i < half ? i + half - 1 : i - half; };  // ascending index -> bin-order index
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        for (int k = threadIdx.x; k < K; k += blockDim.x) s_row[k] = ls[row * K + k];
        __syncthreads();
        for (int u = 0; u < U; ++u) {
            float2* o = out + u * user_stride + row * K;
            for (int k = threadIdx.x; k < K; k += blockDim.x) {
                const int i = k + half < K ? k + half : k + half - K;
                float2 v;
                if (i <= u) {
                    v = s_row[bin(u)];  // own first pilot, or below it: held
                } else {
                    const int p0 = i - (i - u) % U, p1 = p0 + U;
                    if (p0 == i || p1 >= K) {
                        v = s_row[bin(p0)];  // own pilot, or above the last one: held
                    } else {
                        const float w = (float)(phi(i) - phi(p0)) / (float)(phi(p1) - phi(p0));
                        const float2 a = s_row[bin(p0)], b = s_row[bin(p1)];
                        v = make_float2(fmaf(w, b.x - a.x, a.x), fmaf(w, b.y - a.y, a.y));
                    }
                }
                o[k] = v;
            }
        }
        __syncthreads();  // the row buffer is refilled next
    }
}

// Teams take items (frame f, user group g, data symbol s), consecutive items sharing (f, g) so that the teams working
// at the same time read the same detector rows (L1/L2).  Outputs: combined [F][S-P][U][K] ascending frequency, bits
// [F][S-P][U][row], P pilot symbols (U time-orthogonal, 1 comb).  p.first_sym = P, p.n_sym_work = S-P; n_users = U,
// UP = groups * UG.
// SOFT: also p.llr [F][S-P][U][K][b] from soft_tab [F][U][K] (k_mu_soft_scale); the hard kernel ignores soft_tab.
template <class PL, int UG, bool SOFT = false>
__global__ void __launch_bounds__(PL::THREADS, 1) lsmrc_mu_data(const KernelParams p, const float2* __restrict__ wd, int n_users, int n_groups,
                                                                const float2* __restrict__ soft_tab)
{
    constexpr int N = PL::N, P = PL::P, T = PL::T, K = N - 1;
    extern __shared__ __align__(16) float2 smem[];
    float2* s_tw1 = smem;
    float2* s_tw2 = smem + PL::TW1;
    float2* s_tiles = smem + PL::TWN;
    const int team = threadIdx.x / T;
    const int t = threadIdx.x % T;
    float2* my_tiles = s_tiles + team * PL::TEAM_STRIDE;
    for (int i = threadIdx.x; i < PL::TWN; i += PL::THREADS) smem[i] = p.twiddles[i];
    __syncthreads();

    const int U = n_users, UP = n_groups * UG, D = p.n_sym_work;
    const long long n_items = (long long)p.n_frames * n_groups * D;
    const long long n_rounds = (n_items + (long long)gridDim.x * PL::TEAMS - 1) / ((long long)gridDim.x * PL::TEAMS);
    for (long long r = 0; r < n_rounds; ++r) {  // every team runs the same number of rounds: team_sync stays uniform
        const long long raw = (r * gridDim.x + blockIdx.x) * PL::TEAMS + team;
        const bool ok = raw < n_items;
        const long long item = ok ? raw : n_items - 1;
        const int s = (int)(item % D);
        const long long fg = item / D;
        const int g = (int)(fg % n_groups);
        const long long f = fg / n_groups;
        const float2* x0 = p.rx + f * p.frame_stride + (long long)(p.first_sym + s) * p.sym_stride + p.cp;
        const float2* w0 = wd + (f * UP + (long long)g * UG) * p.n_ant * N;
        const long long wstride = (long long)p.n_ant * N;  // between users
        float2 acc[UG][P];
#pragma unroll
        for (int j = 0; j < UG; ++j)
#pragma unroll
            for (int sl = 0; sl < P; ++sl) acc[j][sl] = make_float2(0.f, 0.f);
        for (int a = 0; a < p.n_ant; ++a) {
            float2 v[P];
            row_load<PL>(v, x0 + (long long)a * p.ant_stride, t);
            float2* tile = my_tiles + (PL::NBUF == 2 ? (a & 1) * PL::TILE : 0);
            const float2* wa = w0 + (long long)a * N;
            row_fft<PL>(v, nullptr, tile, s_tw1, s_tw2, t, team, [&](int sl, int bin, float2 y) {
                const int hp = PL::hpos(sl, t, bin);
#pragma unroll
                for (int j = 0; j < UG; ++j) acc[j][sl] = cmac(acc[j][sl], y, __ldg(wa + j * wstride + hp));
            });
        }
        // epilogue per user: ascending-frequency store, hard demap into the team's tile (bytes), bit packing; SOFT: max-log
        // LLRs of the user's symbol times scale, at rho (DESIGN.md 8f).  BC = bits per symbol, fixed at compile time for
        // the soft epilogue (straight-line soft_symbol); 0 = p.qam_bits at run time (the hard kernel).
        uint8_t* s_idx = reinterpret_cast<uint8_t*>(my_tiles);
        auto epilogue = [&](auto bconst) {
            constexpr int BC = decltype(bconst)::value;
            const int b = BC > 0 ? BC : p.qam_bits;
#pragma unroll
            for (int j = 0; j < UG; ++j) {
                // padding users of the last group: teams of whole warps skip them; narrower teams share a warp's
                // __syncwarp with teams of other groups, so they run the epilogue without storing and every lane passes
                // the same barriers
                const int u = g * UG + j;
                if constexpr (PL::T >= 32) {
                    if (u >= U) break;
                }
                const bool store = ok && u < U;
                const long long orow = (f * D + s) * U + (u < U ? u : U - 1);
                float2* out_row = p.combined + orow * K;
                [[maybe_unused]] const float2* tab_row = SOFT ? soft_tab + (f * U + u) * K - 1 : nullptr;  // indexed by bin
                [[maybe_unused]] float* llr_row = SOFT ? p.llr + orow * K * BC : nullptr;
                team_sync<PL>(team);  // the tile (last row's exchange buffer, or the previous user's bytes) is free
#pragma unroll
                for (int sl = 0; sl < P; ++sl) {
                    const int bin = PL::bin_of(sl, t);
                    if (bin > 0) {
                        const int pos = (bin < N / 2) ? (bin - 1 + N / 2) : (bin - N / 2);
                        if (store) out_row[pos] = acc[j][sl];
                        s_idx[pos] = (uint8_t)demap_symbol(acc[j][sl].x, acc[j][sl].y, b);
                        if constexpr (SOFT) {
                            if (store) {
                                const float2 rs = __ldg(tab_row + bin);  // (rho, scale)
                                float l[BC];
                                soft_symbol<BC>(__fmul_rn(acc[j][sl].x, rs.y), __fmul_rn(acc[j][sl].y, rs.y), rs.x, l);
#pragma unroll
                                for (int q = 0; q < BC; ++q) llr_row[pos * BC + q] = l[q];
                            }
                        }
                    }
                }
                if (p.bits != nullptr) {
                    team_sync<PL>(team);
                    pack_bits<PL>(s_idx, p.bits + orow * p.bits_row_bytes, p.bits_row_bytes, b, store, t);
                }
            }
        };
        if constexpr (SOFT) {
            if (p.qam_bits == 2) epilogue(std::integral_constant<int, 2>{});
            else if (p.qam_bits == 4) epilogue(std::integral_constant<int, 4>{});
            else epilogue(std::integral_constant<int, 6>{});
        } else {
            epilogue(std::integral_constant<int, 0>{});
        }
        team_sync<PL>(team);  // the bytes alias the tile the next item's first row is exchanged through
    }
}

// ---- multi-user downlink (DESIGN.md 8g) ------------------------------------------------------------------------
// Reciprocal ZF / regularised-ZF precoder from the uplink estimate: P_k[a][u] = W_k[u][a] = conj(Hzf[k][u][a])
// (k_zf_create on X = conj(H) with lambda = reg), laid out by k_mu_weights<PL, true> in plain bin order [F][U][A][N].
// One common gain per frame, g_f = sqrt(U*K / sum_k |P_k|_F^2), |P_k|_F = |Hzf_k|_F.

// Power, step 1: part[f * n_chunks + c] = sum of |x|^2 over elements [c*chunk, (c+1)*chunk) of frame f's block of
// frame_elems.  Fixed reduction order (per-thread strided sums, warp shuffles, warps in order): deterministic.
__global__ void k_sq_norm_chunks(const float2* __restrict__ x, long long frame_elems, int chunk, int n_chunks, float* __restrict__ part)
{
    const long long f = blockIdx.x / n_chunks;
    const long long i0 = (long long)(blockIdx.x - f * n_chunks) * chunk;
    const int n = (int)min((long long)chunk, frame_elems - i0);
    const float2* p = x + f * frame_elems + i0;
    float acc = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float2 v = p[i];
        acc += v.x * v.x + v.y * v.y;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    __shared__ float s_w[32];
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) t += s_w[w];
        part[blockIdx.x] = t;
    }
}

// Power, step 2: gain[f] = sqrt(target / sum_c part[f][c]), one warp per frame, fixed order.  A frame whose precoder is
// zero on every subcarrier (all singular) gets gain 0.
__global__ void k_dl_gain(const float* __restrict__ part, int n_chunks, int n_frames, float target, float* __restrict__ gain)
{
    const int f = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (f >= n_frames) return;
    const int lane = threadIdx.x & 31;
    float acc = 0.f;
    for (int c = lane; c < n_chunks; c += 32) acc += part[(long long)f * n_chunks + c];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) gain[f] = acc > 0.f ? sqrtf(target / acc) : 0.f;
}

// Precoding, inverse FFT and cyclic prefix, fused.  Teams take items (frame f, downlink symbol d, antenna a), a fastest,
// so that the teams running at the same time share (f, d) and read the same symbol rows out of L1/L2.  Per item the
// team forms the transform's input in registers -- slot n1 of thread t holds bin n = n1*T + t, row_load's natural order:
//   v = conj(z[n]),  z[n] = sum_u P[u][a][n] * s[u][asc(n)],  z[0] = 0
// -- runs the FORWARD row transform, IDFT(z) = conj(DFT(conj z)) / N, and the sink writes g/N * conj(Y) for time index
// n = bin_of(sl, t) at C + n, and again at n - (N - C) when n >= N - C (the cyclic prefix).  On the shuffle-stage plans
// the sink sees y' = u * Y, slots out of order: Y = Plan::unfix(y'), and bin_of gives the index (DESIGN.md 8g).
// pd [F][U][A][N] bin order; sym [F][Sd][U][K] ascending frequency; gain [F]; tx [F][Sd][A][N+C], CP first.
constexpr int kDlMinBlocks = 3;  // resident CTAs per SM the precode kernel is compiled for (168 registers at four warps)

template <class PL>
__global__ void __launch_bounds__(PL::THREADS, kDlMinBlocks) lsmrc_dl_precode(const float2* __restrict__ pd, const float2* __restrict__ sym,
                                                                   const float* __restrict__ gain, float2* __restrict__ tx,
                                                                   const float2* __restrict__ twiddles, int n_frames, int n_sym,
                                                                   int A, int U, int cp)
{
    constexpr int N = PL::N, P = PL::P, T = PL::T, K = N - 1;
    extern __shared__ __align__(16) float2 smem[];
    float2* s_tw1 = smem;
    float2* s_tw2 = smem + PL::TW1;
    float2* s_tiles = smem + PL::TWN;
    const int team = threadIdx.x / T;
    const int t = threadIdx.x % T;
    float2* my_tiles = s_tiles + team * PL::TEAM_STRIDE;
    for (int i = threadIdx.x; i < PL::TWN; i += PL::THREADS) smem[i] = twiddles[i];
    __syncthreads();

    const long long n_items = (long long)n_frames * n_sym * A;
    const long long n_rounds = (n_items + (long long)gridDim.x * PL::TEAMS - 1) / ((long long)gridDim.x * PL::TEAMS);
    for (long long r = 0; r < n_rounds; ++r) {  // every team runs the same number of rounds: team_sync stays uniform
        const long long raw = (r * gridDim.x + blockIdx.x) * PL::TEAMS + team;
        const bool ok = raw < n_items;
        const long long item = ok ? raw : n_items - 1;
        const int a = (int)(item % A);
        const long long fd = item / A;  // f * Sd + d
        const long long f = fd / n_sym;
        const float2* s_row = sym + fd * U * K;
        const float2* p_row = pd + (f * U * A + a) * N;
        float2 v[P];
#pragma unroll
        for (int n1 = 0; n1 < P; ++n1) v[n1] = make_float2(0.f, 0.f);
        for (int u = 0; u < U; ++u) {
            const float2* pu = p_row + (long long)u * A * N;
            const float2* su = s_row + (long long)u * K;
#pragma unroll
            for (int n1 = 0; n1 < P; ++n1) {
                const int n = n1 * T + t;
                if (n > 0) v[n1] = cmac(v[n1], __ldg(pu + n), __ldg(su + (n < N / 2 ? n - 1 + N / 2 : n - N / 2)));
            }
        }
#pragma unroll
        for (int n1 = 0; n1 < P; ++n1) v[n1].y = -v[n1].y;
        const float sc = __ldg(gain + f) * (1.0f / N);  // (exact: N is a power of two)
        float2* out = tx + (fd * A + a) * (N + cp);
        float2* tile = my_tiles + (PL::NBUF == 2 ? (int)(r & 1) * PL::TILE : 0);
        row_fft<PL>(v, nullptr, tile, s_tw1, s_tw2, t, team, [&](int sl, int n, float2 y) {
            const float2 Y = PL::unfix(sl, t, y);
            const float2 o = make_float2(sc * Y.x, -sc * Y.y);
            if (ok) {
                out[cp + n] = o;
                if (n >= N - cp) out[n - (N - cp)] = o;
            }
        });
    }
}

}  // namespace lsmrc
