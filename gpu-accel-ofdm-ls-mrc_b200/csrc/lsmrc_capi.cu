// lsmrc_capi.cu -- the only translation unit that touches CUDA: C ABI of
// include/ofdm_lsmrc.h on top of the fused kernels in lsmrc_kernels.cuh.
//
// Host-side structure (B200-first, not a transliteration of gpuLS.cu):
//  * a handle owns its streams, twiddle tables, staging and pinned result
//    buffers once; nothing is allocated, planned or synchronised per symbol
//    (the reference creates a cuFFT plan and cudaMallocs inside every call and
//    calls cudaDeviceSynchronize after every launch: gpuLS.cu:377-380,452,471);
//  * a frame batch costs two launches (pilot, data) regardless of F, S, A -- one when it is small enough to be
//    launch-latency bound (MODE_ONESHOT);
//  * host-buffer and ring ingest are cut into lanes (stream + staging) so H2D
//    of the next chunk overlaps the kernels and D2H of the previous ones.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ofdm_lsmrc.h"
#include "lsmrc_kernels.cuh"

using namespace lsmrc;

namespace {

struct PlanOps {
    int N, P, R2, R3, teams, threads, twn, minb;
    size_t smem;
    void (*fill_twiddles)(float2*);
    cudaError_t (*prepare)(int* data_ctas_per_sm, int* pilot_ctas_per_sm);
    cudaError_t (*launch)(int mode, const KernelParams&, cudaStream_t, int max_data_ctas);
    // shuffle-stage plans: pilot and data items of whole frames in ONE persistent launch (lsmrc_frames_sh); nullptr otherwise
    cudaError_t (*launch_fused)(const KernelParams&, cudaStream_t, int max_data_ctas);
    // multi-user detection: users per pass of the data kernel, and the launch of the weight layout + data kernel; `soft`
    // selects the kernel with the soft epilogue (soft_tab: k_mu_soft_scale's table; nullptr for the hard one)
    int mu_ug;
    cudaError_t (*mu_prepare)(bool soft, int* ctas_per_sm);
    cudaError_t (*mu_launch)(bool soft, const KernelParams&, const float2* hzf, float2* wd, const float2* soft_tab, int n_users, int max_ctas,
                             int n_sms, cudaStream_t);
    // multi-user downlink: resident CTAs of the precode kernel, and the launch of the bin-order precoder layout + that kernel
    cudaError_t (*dl_prepare)(int* ctas_per_sm);
    cudaError_t (*dl_launch)(const float2* hzf, float2* pd, const float2* sym, const float* gain, float2* tx, const float2* twiddles,
                             int n_frames, int n_sym, int n_ant, int n_users, int cp, int max_ctas, int n_sms, cudaStream_t);
};

// The one-launch kernel (MODE_ONESHOT) of a plan.  Small FFT sizes have a dedicated latency plan:
// more threads per row than the throughput plan, so the serial instruction chain of one thread --
// what a single small frame is bound by -- is several times shorter.
struct OneshotOps {
    int N, P, R2, R3, teams, threads, twn;
    void (*fill_twiddles)(float2*);
    cudaError_t (*prepare)(int smem_optin);
    // antenna split to use for this batch, 0 when the mode does not apply
    int (*split)(int n_frames, int n_sym_work, int n_ant, int n_sms, size_t smem_optin);
    cudaError_t (*launch)(const KernelParams&, cudaStream_t);
};

template <class PL>
void fill_twiddles_impl(float2* tw);

constexpr int kOneshotMaxPilotRounds = 4;
constexpr int kOneshotMinb = 1;  // latency mode: one CTA per SM, the full register file

template <class PL>
size_t oneshot_smem(int n_ant)
{
    return PL::SMEM_BYTES + (size_t)n_ant * PL::N * sizeof(float2) + (size_t)PL::N * sizeof(float);
}

// The one-launch mode pays when the call is launch-latency bound: every CTA repeats the channel
// estimate, so it is used only when that is at most kOneshotMaxPilotRounds rounds of row FFTs, the whole batch fits
// in less than one CTA per SM, and conj(H) of a frame fits in shared memory.
template <class PL>
int oneshot_split_impl(int n_frames, int n_sym_work, int n_ant, int n_sms, size_t smem_optin)
{
    if (n_sym_work < 1) return 0;
    if (oneshot_smem<PL>(n_ant) > smem_optin) return 0;
    if ((n_ant + PL::TEAMS - 1) / PL::TEAMS > kOneshotMaxPilotRounds) return 0;
    int as = 1;
    auto ctas = [&](int a) {
        const int slots = PL::TEAMS / a;
        return (long long)n_frames * ((n_sym_work + slots - 1) / slots);
    };
    if (ctas(1) > n_sms) return 0;
    while (as * 2 <= PL::TEAMS && as * 2 <= n_ant && ctas(as * 2) <= n_sms) as *= 2;
    return as;
}

template <class PL>
cudaError_t oneshot_prepare_impl(int smem_optin)
{
    return cudaFuncSetAttribute(lsmrc_kernel<PL, MODE_ONESHOT, kOneshotMinb>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
}

template <class PL>
cudaError_t oneshot_launch_impl(const KernelParams& p, cudaStream_t st)
{
    const int slots = PL::TEAMS / p.ant_split;
    const unsigned grid = (unsigned)(p.n_frames * ((p.n_sym_work + slots - 1) / slots));
    lsmrc_kernel<PL, MODE_ONESHOT, kOneshotMinb><<<grid, PL::THREADS, oneshot_smem<PL>(p.n_ant), st>>>(p);
    return cudaGetLastError();
}

template <class PL>
OneshotOps make_oneshot_ops()
{
    OneshotOps o;
    o.N = PL::N;
    o.P = PL::P;
    o.R2 = PL::R2;
    o.R3 = PL::R3;
    o.teams = PL::TEAMS;
    o.threads = PL::THREADS;
    o.twn = PL::TWN;
    o.fill_twiddles = &fill_twiddles_impl<PL>;
    o.prepare = &oneshot_prepare_impl<PL>;
    o.split = &oneshot_split_impl<PL>;
    o.launch = &oneshot_launch_impl<PL>;
    return o;
}


template <class PL>
void fill_twiddles_impl(float2* tw)
{
    const double two_pi = 6.283185307179586476925286766559;
    for (int k1 = 1; k1 < PL::P; ++k1)
        for (int t = 0; t < PL::T; ++t) {
            const double ang = -two_pi * (double)(((long long)t * k1) % PL::N) / (double)PL::N;
            // shuffle-stage plans fold Plan::stage1_sign(t) into the inter-stage twiddles
            const double sg = (PL::SH == 2 && (t & 3) == 3) || (PL::SH == 4 && (t & 6) == 6) ? -1.0 : 1.0;
            tw[(k1 - 1) * PL::T + t] = make_float2((float)(sg * cos(ang)), (float)(sg * sin(ang)));
        }
    if (PL::SH > 1)  // W_T^(q*k2) per lane position q: [16 register pairs j][SH] x (register 2j, register 2j+1), see sh_load_twiddles
        for (int j = 0; j < 16; ++j)
            for (int q = 0; q < PL::SH; ++q) {
                const int hi = PL::SH == 2 ? q : (q >> 1);
                int kk = 0;  // 5-bit reversal of 2j
                for (int b = 0; b < 5; ++b)
                    if ((2 * j) & (1 << b)) kk |= 1 << (4 - b);
                for (int c = 0; c < 2; ++c) {
                    const int k2 = kk + 16 * (hi ^ c);
                    const double ang = -two_pi * (double)((q * k2) % PL::T) / (double)PL::T;
                    tw[PL::TW1 + (j * PL::SH + q) * 2 + c] = make_float2((float)cos(ang), (float)sin(ang));
                }
            }
    if (PL::R3 > 1)
        for (int k2 = 1; k2 < PL::R2; ++k2)
            for (int m2 = 0; m2 < PL::R3; ++m2) {
                const double ang = -two_pi * (double)((m2 * k2) % PL::T) / (double)PL::T;
                tw[PL::TW1 + (k2 - 1) * PL::R3 + m2] = make_float2((float)cos(ang), (float)sin(ang));
            }
}

// the pilot kernel keeps the pilot, 1/|X|^2 and the energy partials of its P bins in registers on
// top of the FFT working set: give the 32-point plans a 255-register budget there
template <class PL, int MINB>
constexpr int pilot_minb() { return (PL::P >= 32 && MINB > 2) ? 2 : MINB; }

// dynamic shared memory of lsmrc_data_sh: per team one channel row and a tile
template <class PL>
constexpr size_t data_sh_smem() { return sizeof(float2) * (size_t)(PL::TEAMS * (PL::N + PL::TILE)); }

// Resident CTAs per SM of a kernel that allocates `tmem_cols` tensor-memory columns per CTA.  The runtime's occupancy
// calculator answers 1 for any such kernel (it cannot know how many of the SM's 512 columns a CTA takes), so the
// limits are applied by hand: registers (allocated per warp in units of 256), shared memory (dynamic + static + 1 KB
// reserved per CTA), warps, and columns.
template <class K>
cudaError_t occupancy_with_tmem(int* ctas_per_sm, K kernel, int threads, size_t dyn_smem, int tmem_cols)
{
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
    if (e != cudaSuccess) return e;
    int dev = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    int regs_sm = 0, smem_sm = 0, threads_sm = 0;
    if ((e = cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&threads_sm, cudaDevAttrMaxThreadsPerMultiProcessor, dev)) != cudaSuccess) return e;
    const int warps = (threads + 31) / 32;
    const int regs_warp = ((fa.numRegs * 32 + 255) / 256) * 256;
    int n = regs_sm / (regs_warp * warps);
    const size_t smem_cta = dyn_smem + fa.sharedSizeBytes + 1024;
    if ((int)((size_t)smem_sm / smem_cta) < n) n = (int)((size_t)smem_sm / smem_cta);
    if (threads_sm / threads < n) n = threads_sm / threads;
    if (tmem_cols > 0 && 512 / tmem_cols < n) n = 512 / tmem_cols;
    *ctas_per_sm = n;
    return cudaSuccess;
}

// dynamic shared memory of lsmrc_pilot_sh: the LS-divide table (one row) and a tile per team
template <class PL>
constexpr size_t pilot_sh_smem() { return sizeof(float2) * (size_t)(PL::N + PL::TEAMS * PL::TILE); }

template <class PL, int MINB>
cudaError_t prepare_impl(int* data_ctas_per_sm, int* pilot_ctas_per_sm)
{
    cudaError_t e = cudaFuncSetAttribute(lsmrc_kernel<PL, MODE_PILOT, pilot_minb<PL, MINB>()>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PL::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(lsmrc_kernel<PL, MODE_DATA, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)PL::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(lsmrc_kernel<PL, MODE_FFT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)PL::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    // resident CTAs per SM: the persistent data grid is this times the SM count; the pilot grid is
    // sized to at most one such wave when frames are few
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(pilot_ctas_per_sm, lsmrc_kernel<PL, MODE_PILOT, pilot_minb<PL, MINB>()>,
                                                      PL::THREADS, PL::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    // (tensor-memory columns per CTA: 2P for the stage-1 twiddles, power of two >= 32)
    e = occupancy_with_tmem(data_ctas_per_sm, lsmrc_kernel<PL, MODE_DATA, MINB>, PL::THREADS, PL::SMEM_BYTES, PL::TW_TMEM ? 2 * PL::P : 0);
    if (e != cudaSuccess) return e;
    if constexpr (PL::X_TMA) {  // the bulk-copy instantiation of the data kernel shares the persistent grid size
        e = cudaFuncSetAttribute(lsmrc_kernel<PL, MODE_DATA, MINB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PL::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        int xt = 0;
        e = occupancy_with_tmem(&xt, lsmrc_kernel<PL, MODE_DATA, MINB, true>, PL::THREADS, PL::SMEM_BYTES, PL::TW_TMEM ? 2 * PL::P : 0);
        if (e != cudaSuccess) return e;
        if (xt < *data_ctas_per_sm) *data_ctas_per_sm = xt;
    }
    if constexpr (PL::SH > 1) {
        // shuffle-stage plans: large batches run the dedicated data kernel (the generic one serves the antenna-split
        // launches of tiny batches); both share the persistent grid size
        e = cudaFuncSetAttribute(lsmrc_data_sh<PL, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)data_sh_smem<PL>());
        if (e != cudaSuccess) return e;
        int sh = 0;
        e = occupancy_with_tmem(&sh, lsmrc_data_sh<PL, MINB>, PL::THREADS, data_sh_smem<PL>(), 128);
        if (e != cudaSuccess) return e;
        if (sh < *data_ctas_per_sm) *data_ctas_per_sm = sh;
        // ... and the dedicated pilot kernel (batches with one antenna group per frame or more)
        e = cudaFuncSetAttribute(lsmrc_pilot_sh<PL, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pilot_sh_smem<PL>());
        if (e != cudaSuccess) return e;
        e = occupancy_with_tmem(pilot_ctas_per_sm, lsmrc_pilot_sh<PL, MINB>, PL::THREADS, pilot_sh_smem<PL>(), 128);
        if (e != cudaSuccess) return e;
        // ... and both in one launch (whole frames, batches large enough for one team per (frame, symbol) pair)
        e = cudaFuncSetAttribute(lsmrc_frames_sh<PL, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)data_sh_smem<PL>());
        if (e != cudaSuccess) return e;
        e = occupancy_with_tmem(&sh, lsmrc_frames_sh<PL, MINB>, PL::THREADS, data_sh_smem<PL>(), 128);
        if (e != cudaSuccess) return e;
        if (sh < *data_ctas_per_sm) *data_ctas_per_sm = sh;
    }
    return cudaSuccess;
}

// pilot + data items of whole frames on one ticket counter (shuffle-stage plans)
template <class PL, int MINB>
cudaError_t launch_fused_impl(const KernelParams& p, cudaStream_t st, int max_data_ctas)
{
    if constexpr (PL::SH > 1) {
        const long long items = (long long)p.n_frames * p.n_groups + ((long long)p.n_frames * p.n_sym_work + PL::TEAMS - 1) / PL::TEAMS;
        const unsigned grid = (unsigned)(items < max_data_ctas ? items : max_data_ctas);
        lsmrc_frames_sh<PL, MINB><<<grid, PL::THREADS, data_sh_smem<PL>(), st>>>(p);
        return cudaGetLastError();
    } else {
        (void)p, (void)st, (void)max_data_ctas;
        return cudaErrorNotSupported;
    }
}

template <class PL, int MINB>
cudaError_t launch_impl(int mode, const KernelParams& p, cudaStream_t st, int max_data_ctas)
{
    if (mode == MODE_FFT) {
        const long long groups = ((long long)p.n_frames + PL::TEAMS - 1) / PL::TEAMS;
        const unsigned grid = (unsigned)(groups < 4 * (long long)max_data_ctas ? groups : 4 * (long long)max_data_ctas);
        lsmrc_kernel<PL, MODE_FFT, MINB><<<grid, PL::THREADS, PL::SMEM_BYTES, st>>>(p);
    } else if (mode == MODE_PILOT) {
        const long long n_virtual = (long long)((p.n_frames + p.frames_per_cta - 1) / p.frames_per_cta) * p.n_groups;
        const long long cap = p.pilot_grid_cap > 0 ? p.pilot_grid_cap : n_virtual;
        const unsigned grid = (unsigned)(n_virtual < cap ? n_virtual : cap);  // CTAs stride over the virtual CTAs
        if constexpr (PL::SH > 1) {
            if (p.frames_per_cta == 1) {
                lsmrc_pilot_sh<PL, MINB><<<grid, PL::THREADS, pilot_sh_smem<PL>(), st>>>(p);
                return cudaGetLastError();
            }
        }
        lsmrc_kernel<PL, MODE_PILOT, pilot_minb<PL, MINB>()><<<grid, PL::THREADS, PL::SMEM_BYTES, st>>>(p);
    } else {
        long long items;
        KernelParams q = p;
        if (PL::H_RING) {
            items = (long long)p.n_frames * ((p.n_sym_work + PL::TEAMS - 1) / PL::TEAMS);
            q.ant_split = 1;
        } else {
            // few (frame, symbol) pairs: split each pair's antennas over several teams of a CTA so that
            // more of the GPU works on the batch (single-frame latency); many pairs: one team per pair
            const long long n_work = (long long)p.n_frames * p.n_sym_work;
            int as = 1;
            while (as * 2 <= PL::TEAMS && as * 2 <= p.n_ant &&
                   (n_work * (as * 2) + PL::TEAMS - 1) / PL::TEAMS <= (long long)max_data_ctas / 2)
                as *= 2;
            q.ant_split = as;
            const int slots = PL::TEAMS / as;
            items = (n_work + slots - 1) / slots;
        }
        const unsigned grid = (unsigned)(items < max_data_ctas ? items : max_data_ctas);  // persistent CTAs
        if constexpr (PL::SH > 1) {
            if (q.ant_split == 1) {
                lsmrc_data_sh<PL, MINB><<<grid, PL::THREADS, data_sh_smem<PL>(), st>>>(q);
                return cudaGetLastError();
            }
        }
        if constexpr (PL::X_TMA) {
            if (q.x_tma) {  // rows 16-byte aligned: the instantiation that brings them in by bulk copy
                lsmrc_kernel<PL, MODE_DATA, MINB, true><<<grid, PL::THREADS, PL::SMEM_BYTES, st>>>(q);
                return cudaGetLastError();
            }
        }
        lsmrc_kernel<PL, MODE_DATA, MINB><<<grid, PL::THREADS, PL::SMEM_BYTES, st>>>(q);
    }
    return cudaGetLastError();
}

// Multi-user data kernel (lsmrc_mu_data): users per pass.  Each thread keeps UG * P complex sums in registers next to the
// FFT working set: the most that compiles without spills (-Xptxas -v) -- two users for the 32-point plans of 1024 and
// 4096 points (128 registers of sums), one for 512 and 2048 (two spill there), four at 16 points, eight at 8.  Larger
// U re-runs the row transforms once per group of UG users (DESIGN.md 8e).  The soft epilogue (SOFT) compiles without
// spills at the same UG on every plan (DESIGN.md 8f).
template <class PL>
constexpr int mu_ug() { return PL::P >= 32 ? ((PL::N == 512 || PL::N == 2048) ? 1 : 2) : (PL::P >= 16 ? 4 : 8); }

template <class PL>
constexpr size_t mu_smem() { return sizeof(float2) * (size_t)(PL::TWN + PL::TEAMS * PL::TEAM_STRIDE); }

template <class PL>
cudaError_t mu_prepare_impl(bool soft, int* ctas_per_sm)
{
    constexpr int UG = mu_ug<PL>();
    const auto kernel = soft ? lsmrc_mu_data<PL, UG, true> : lsmrc_mu_data<PL, UG, false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mu_smem<PL>());
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, kernel, PL::THREADS, mu_smem<PL>());
}

// max_ctas: resident CTAs of the (hard or soft) lsmrc_mu_data on the whole GPU (mu_prepare_impl x SMs)
template <class PL>
cudaError_t mu_launch_impl(bool soft, const KernelParams& p, const float2* hzf, float2* wd, const float2* soft_tab, int n_users, int max_ctas,
                           int n_sms, cudaStream_t st)
{
    constexpr int UG = mu_ug<PL>();
    const int groups = (n_users + UG - 1) / UG;
    cudaError_t e;
    const long long rows = (long long)p.n_frames * groups * UG * p.n_ant;
    long long wblocks = (rows * PL::N + 255) / 256;
    if (wblocks > (long long)n_sms * 16) wblocks = (long long)n_sms * 16;
    k_mu_weights<PL><<<(unsigned)wblocks, 256, 0, st>>>(hzf, wd, p.n_ant, n_users, groups * UG, rows);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const long long items = (long long)p.n_frames * groups * p.n_sym_work;
    long long grid = (items + PL::TEAMS - 1) / PL::TEAMS;
    if (grid > max_ctas) grid = max_ctas;
    if (soft) lsmrc_mu_data<PL, UG, true><<<(unsigned)grid, PL::THREADS, mu_smem<PL>(), st>>>(p, wd, n_users, groups, soft_tab);
    else lsmrc_mu_data<PL, UG, false><<<(unsigned)grid, PL::THREADS, mu_smem<PL>(), st>>>(p, wd, n_users, groups, soft_tab);
    return cudaGetLastError();
}

// the precode kernel (lsmrc_dl_precode) has the multi-user data kernel's shared-memory layout: twiddles and team tiles
template <class PL>
cudaError_t dl_prepare_impl(int* ctas_per_sm)
{
    cudaError_t e = cudaFuncSetAttribute(lsmrc_dl_precode<PL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mu_smem<PL>());
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, lsmrc_dl_precode<PL>, PL::THREADS, mu_smem<PL>());
}

// max_ctas: resident CTAs of lsmrc_dl_precode on the whole GPU (dl_prepare_impl x SMs)
template <class PL>
cudaError_t dl_launch_impl(const float2* hzf, float2* pd, const float2* sym, const float* gain, float2* tx, const float2* twiddles,
                           int n_frames, int n_sym, int n_ant, int n_users, int cp, int max_ctas, int n_sms, cudaStream_t st)
{
    const long long rows = (long long)n_frames * n_users * n_ant;
    long long wblocks = (rows * PL::N + 255) / 256;
    if (wblocks > (long long)n_sms * 16) wblocks = (long long)n_sms * 16;
    // (plans without a shuffle stage: their slot layout is bin order, the uplink's instantiation serves)
    k_mu_weights<PL, (PL::SH > 1)><<<(unsigned)wblocks, 256, 0, st>>>(hzf, pd, n_ant, n_users, n_users, rows);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long items = (long long)n_frames * n_sym * n_ant;
    long long grid = (items + PL::TEAMS - 1) / PL::TEAMS;
    if (grid > max_ctas) grid = max_ctas;
    lsmrc_dl_precode<PL><<<(unsigned)grid, PL::THREADS, mu_smem<PL>(), st>>>(pd, sym, gain, tx, twiddles, n_frames, n_sym, n_ant, n_users, cp);
    return cudaGetLastError();
}

template <class PL, int MINB>
PlanOps make_ops()
{
    PlanOps o;
    o.N = PL::N;
    o.P = PL::P;
    o.R2 = PL::R2;
    o.R3 = PL::R3;
    o.teams = PL::TEAMS;
    o.threads = PL::THREADS;
    o.twn = PL::TWN;
    o.minb = MINB;
    o.smem = PL::SMEM_BYTES;
    o.fill_twiddles = &fill_twiddles_impl<PL>;
    o.prepare = &prepare_impl<PL, MINB>;
    o.launch = &launch_impl<PL, MINB>;
    o.launch_fused = PL::SH > 1 ? &launch_fused_impl<PL, MINB> : nullptr;
    o.mu_ug = mu_ug<PL>();
    o.mu_prepare = &mu_prepare_impl<PL>;
    o.mu_launch = &mu_launch_impl<PL>;
    o.dl_prepare = &dl_prepare_impl<PL>;
    o.dl_launch = &dl_launch_impl<PL>;
    return o;
}

// ---- the plans.  Template arguments: N, P (points per thread), R2, R3, teams per CTA, tile buffers per team, rows of
// x prefetched to L2, rows of Hconj prefetched to L1, register prefetch of the next row, Hconj ring,
// x rows by bulk copy, stage-1 twiddles in tensor memory, lanes of the shuffle stage.  Each setting is the measured
// winner of its A/B (DESIGN.md section 3 keeps the log, including the variants that lost and were deleted).
// (64 points: 8 threads x 8 points per row.  16 x 4 -- teams of 4 threads reading 32 contiguous bytes per load, 8 lines per
// warp request -- measured 13-17 % slower: c1 3.15 -> 3.6 TB/s, 16 antennas 3.7 -> 4.3, 64 antennas 3.9 -> 4.6)
using Plan64 = Plan<64, 8, 8, 1, 8, 2, 1, 1, 0>;  // (next sample row prefetched to L2, next channel row to L1: +1..4 % over the register prefetch;
                                                  // 8 teams per CTA: the pilot kernel of 16-antenna frames 0.042 -> 0.034 ms, the rest +-1 %)
using Plan128 = Plan<128, 16, 8, 1, 16, 2, 0, 0, 1>;  // (8 x 4 x 4, three stages with 128-byte team loads: 25-30 % slower; L2/L1 prefetches: -1..-9 %)
using Plan256 = Plan<256, 16, 16, 1, 8, 2, 1, 1, 1>;  // (+ L2 prefetch of the sample row after next: +7 %)
using Plan512 = Plan<512, 32, 16, 1, 8, 1, 1, 1>;  // (tensor-memory twiddles measured 10 % slower here: teams of 16 threads)
using Plan1024 = Plan<1024, 32, 32, 1, 4, 1, 0, 1, 0, true, true, true>;
using Plan2048 = Plan<2048, 32, 32, 1, 2, 1, 1, 0, 0, false, false, true, 2>;
using Plan4096 = Plan<4096, 32, 32, 1, 1, 1, 1, 0, 0, false, false, true, 4>;
constexpr int kMinBlocks = 3;  // 3 CTAs (12 warps) per SM at 168 registers: measured best for every size

// LSMRC_ONLY_N=<size> (development): instantiate the kernels of one FFT size only -- a full build takes 85 s
#ifdef LSMRC_ONLY_N
#define LSMRC_HAVE(n) ((n) == LSMRC_ONLY_N)
#else
#define LSMRC_HAVE(n) 1
#endif

// One plan per FFT size (64..4096).  N/P threads own a row; see lsmrc_kernels.cuh.
const PlanOps* find_plan(int N)
{
    static const PlanOps plans[] = {
#if LSMRC_HAVE(64)
        make_ops<Plan64, kMinBlocks>(),
#endif
#if LSMRC_HAVE(128)
        make_ops<Plan128, kMinBlocks>(),
#endif
#if LSMRC_HAVE(256)
        make_ops<Plan256, kMinBlocks>(),
#endif
#if LSMRC_HAVE(512)
        make_ops<Plan512, kMinBlocks>(),
#endif
#if LSMRC_HAVE(1024)
        make_ops<Plan1024, kMinBlocks>(),
#endif
#if LSMRC_HAVE(2048)
        make_ops<Plan2048, kMinBlocks>(),
#endif
#if LSMRC_HAVE(4096)
        make_ops<Plan4096, kMinBlocks>(),
#endif
    };
    for (const PlanOps& o : plans)
        if (o.N == N) return &o;
    return nullptr;
}

// One-launch kernels.  64..256 points get a latency plan (8 points per thread instead of 16: a
// thread's serial chain is what bounds a single small frame); larger sizes reuse the throughput plan.
const OneshotOps* find_oneshot_plan(int N)
{
    static const OneshotOps plans[] = {
#if LSMRC_HAVE(64)
        make_oneshot_ops<Plan<64, 8, 8, 1, 16, 2>>(),
#endif
#if LSMRC_HAVE(128)
        make_oneshot_ops<Plan<128, 8, 4, 4, 16, 1>>(),
#endif
#if LSMRC_HAVE(256)
        make_oneshot_ops<Plan<256, 8, 8, 4, 8, 1>>(),
#endif
#if LSMRC_HAVE(512)
        make_oneshot_ops<Plan512>(),
#endif
#if LSMRC_HAVE(1024)
        make_oneshot_ops<Plan1024>(),
#endif
#if LSMRC_HAVE(2048)
        make_oneshot_ops<Plan2048>(),
#endif
#if LSMRC_HAVE(4096)
        make_oneshot_ops<Plan4096>(),
#endif
    };
    for (const OneshotOps& o : plans)
        if (o.N == N) return &o;
    return nullptr;
}

// device-side channel state for a batch of frames (internal layouts, see KernelParams)
struct ChanState {
    float2* hwork = nullptr;          // [frames][A][N]
    float* hsqrd = nullptr;           // [frames][K]
    float* epart = nullptr;           // [frames + kPilotCtaTarget][N]
    unsigned int* counters = nullptr; // [frames], zero between launches
    unsigned long long* ticket = nullptr;  // data-kernel work-item counter + departed-CTA counter (self-resetting), [2] launch number of the fused kernel
    unsigned int* ready = nullptr;         // [frames] fused kernel: launch number that last completed the frame's channel state
    int frames = 0;
};
constexpr int kPilotCtaTarget = 4096;  // upper bound on frames*groups - frames (epart scratch rows)

struct Lane {
    ChanState ch;
    cudaStream_t st = nullptr;
    cudaEvent_t copied = nullptr, done = nullptr;
    cudaEvent_t t_start = nullptr, t_kernels = nullptr;  // timeline of the ring path (lsmrc_ring_trace): submission enqueued, kernels finished
    float2* d_rx = nullptr;     // [max_frames][S][A][N+C]
    short2* d_rx16 = nullptr;   // the same frames in the radio's wire format (int16 I/Q), allocated by the first sc16 call
    float2* d_hconj = nullptr;  // [max_frames][A][K] (reference layout, only when the caller wants it back)
    float2* d_comb = nullptr;   // [max_frames][S-1][K]
    uint8_t* d_bits = nullptr;  // [max_frames][S-1][row]
    // pinned result buffers of the ring path (max_frames frames)
    float2* h_comb = nullptr;
    uint8_t* h_bits = nullptr;
    float2* h_hconj = nullptr;
    // device-visible aliases of the three pinned buffers (in-place ring path)
    float2* a_comb = nullptr;
    uint8_t* a_bits = nullptr;
    float2* a_hconj = nullptr;
    bool busy = false;
    int ring_frames = 0;  // frames of the submission in flight on this lane
};

std::mutex g_err_mutex;
std::string g_create_error;

}  // namespace

struct lsmrc_ctx {
    lsmrc_config cfg;
    int K = 0;
    size_t row_bytes = 0;
    size_t slot_elems = 0;   // A*(N+C)
    size_t frame_elems = 0;  // S*slot
    const PlanOps* ops = nullptr;
    const OneshotOps* one_ops = nullptr;  // one-launch kernel (own plan, own twiddle table)
    float2* d_one_tw = nullptr;
    int max_data_ctas = 1;  // persistent data-kernel grid: resident CTAs per SM x SM count
    int pilot_wave = 1;     // pilot-kernel CTAs resident at once on the whole GPU
    int n_sms = 1;
    size_t smem_optin = 0;
    long long oneshot_calls = 0;  // batches served by the one-launch kernel
    long long zero_copy_calls = 0;  // ... of which on pinned host buffers in place
    bool oneshot = true;
    bool one_launch_frames = true;  // shuffle-stage plans: pilot and data items of large batches in one persistent launch (lsmrc_frames_sh)
    long long fused_calls = 0;
    bool zero_copy = true;        // one-launch kernel reads/writes pinned host buffers in place (small frames)
    bool h2d_strip_cp = true;     // lsmrc_demod_frames_host: strided H2D copy that leaves the cyclic prefix behind
    size_t h2d_strip_min_row = 512;   // ... for rows of at least this many bytes (LSMRC_H2D_STRIP_MIN_ROW, 0 = off);
                                      // measured: +6 % at 8 KB rows, +12 % at 2 KB and still +5..12 % at 512 B rows
    float2* d_tw = nullptr;
    float2* d_pilot_bin = nullptr;
    bool have_pilot = false;
    cudaStream_t own_stream = nullptr;
    cudaStream_t user_stream = nullptr;
    bool use_user_stream = false;
    // channel state of the device-resident path
    ChanState dev_ch;
    // per-symbol path state (one frame)
    ChanState one_ch;
    float2* d_sym = nullptr;
    float2* d_one_hconj = nullptr;
    float2* d_one_comb = nullptr;
    uint8_t* d_one_bits = nullptr;
    float2* h_one_sym = nullptr;   // pinned staging for pageable ring slots
    float2* h_one_comb = nullptr;  // pinned
    uint8_t* h_one_bits = nullptr;
    bool have_channel = false;
    std::vector<Lane> lanes;
    cudaEvent_t ring_epoch = nullptr;     // time zero of lsmrc_ring_trace: the first ring submission of the handle
    unsigned long long* d_hit = nullptr;  // frame-sync first-hit key
    float* d_noise_part = nullptr;        // [frames][S-1] row partials of the noise estimator
    size_t noise_part_rows = 0;
    // multi-user path (lsmrc_demod_frames_device_mu): its own channel state and scratch, grown on demand
    ChanState mu_ch;
    float2* d_mu_hconj = nullptr;  // [U][F][A][K] conj(H) per user, as the pilot kernel writes it
    float2* d_mu_ls = nullptr;     // comb pilots: [F][A][K] LS estimate of pilot symbol 0, input of k_mu_comb_interp
    float2* d_mu_hzf = nullptr;    // [F][K][U][A] conj(W)
    float2* d_mu_wd = nullptr;     // [F][UP][A][N] W in the data kernel's slot layout
    float* d_mu_soft = nullptr;    // soft output: ginv_diag [F][U][K] float, then the (rho, scale) table [F][U][K] float2
    size_t mu_hconj_cap = 0, mu_ls_cap = 0, mu_hzf_cap = 0, mu_wd_cap = 0, mu_soft_cap = 0;  // bytes
    int mu_pilots = LSMRC_MU_PILOTS_TIME;  // frame format of the multi-user calls (lsmrc_set_mu_pilots)
    int* d_mu_count = nullptr;     // singular (frame, subcarrier) pairs
    int mu_max_ctas = 0;           // resident CTAs of the multi-user data kernel (0: not prepared yet)
    int mu_soft_max_ctas = 0;      // the same for its soft instantiation
    // multi-user downlink (lsmrc_precode_frames_device): scratch of its own, so that it never regrows buffers a captured
    // uplink call uses
    float2* d_dl_hzf = nullptr;    // [F][K][U][A] conj(P)
    float2* d_dl_pd = nullptr;     // [F][U][A][N] P in bin order
    float* d_dl_part = nullptr;    // power partials [F][chunks], then the gain [F] when the caller passes none
    size_t dl_hzf_cap = 0, dl_pd_cap = 0, dl_part_cap = 0;  // bytes
    int dl_max_ctas = 0;           // resident CTAs of the precode kernel
    float* soft_llr = nullptr;            // set for the duration of a *_soft call
    float soft_inv_noise = 1.f;
    bool timing = false;
    static constexpr int kEvRing = 256;          // timed calls remembered for lsmrc_kernel_ms_history
    cudaEvent_t ev[kEvRing][3] = {};             // [call % kEvRing] -> {start, after pilot, after data}
    long long ev_calls = 0;                      // timed calls so far
    long long launches = 0;
    std::string err;
};

namespace {

int fail(lsmrc_ctx* h, int code, const std::string& msg)
{
    if (h) h->err = msg;
    else {
        std::lock_guard<std::mutex> g(g_err_mutex);
        g_create_error = msg;
    }
    return code;
}

int fail_cuda(lsmrc_ctx* h, cudaError_t e, const char* what)
{
    return fail(h, LSMRC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CK(h, expr)                                                  \
    do {                                                             \
        cudaError_t _e = (expr);                                     \
        if (_e != cudaSuccess) return fail_cuda((h), _e, #expr);     \
    } while (0)

cudaStream_t compute_stream(lsmrc_ctx* h) { return h->use_user_stream ? h->user_stream : h->own_stream; }

KernelParams base_params(lsmrc_ctx* h)
{
    KernelParams p;
    std::memset(&p, 0, sizeof(p));
    const lsmrc_config& c = h->cfg;
    p.sym_stride = (long long)h->slot_elems;
    p.rx2 = nullptr;
    p.split_sym = 0x7fffffff;
    p.rx_align4 = 0;
    p.frame_stride = (long long)h->frame_elems;
    p.ant_stride = c.fft_size + c.cp_len;
    p.cp = c.cp_len;
    p.n_ant = c.n_ant;
    p.qam_bits = c.qam_bits;
    p.pilot_bin = h->d_pilot_bin;
    p.bits_row_bytes = (int)h->row_bytes;
    p.twiddles = h->d_tw;
    p.llr = h->soft_llr;
    p.inv_noise_var = h->soft_inv_noise;
    return p;
}

int ensure_chan(lsmrc_ctx* h, ChanState& c, int frames, cudaStream_t quiesce)
{
    if (c.frames >= frames) return LSMRC_OK;
    if (quiesce) CK(h, cudaStreamSynchronize(quiesce));
    cudaFree(c.hwork);
    cudaFree(c.hsqrd);
    cudaFree(c.epart);
    cudaFree(c.counters);
    cudaFree(c.ticket);
    cudaFree(c.ready);
    c = ChanState();
    const size_t N = (size_t)h->cfg.fft_size;
    CK(h, cudaMalloc(&c.hwork, (size_t)frames * h->cfg.n_ant * N * sizeof(float2)));
    CK(h, cudaMalloc(&c.hsqrd, (size_t)frames * h->K * sizeof(float)));
    CK(h, cudaMalloc(&c.epart, ((size_t)frames + kPilotCtaTarget) * N * sizeof(float)));
    CK(h, cudaMalloc(&c.counters, (size_t)frames * sizeof(unsigned int)));
    CK(h, cudaMemset(c.counters, 0, (size_t)frames * sizeof(unsigned int)));
    CK(h, cudaMalloc(&c.ticket, 4 * sizeof(unsigned long long)));
    CK(h, cudaMemset(c.ticket, 0, 4 * sizeof(unsigned long long)));
    CK(h, cudaMalloc(&c.ready, (size_t)frames * sizeof(unsigned int)));
    CK(h, cudaMemset(c.ready, 0, (size_t)frames * sizeof(unsigned int)));
    // the memsets run on the legacy stream, the kernels on non-blocking streams that do not order against it
    CK(h, cudaDeviceSynchronize());
    c.frames = frames;
    return LSMRC_OK;
}

void free_chan(ChanState& c)
{
    cudaFree(c.ticket);
    cudaFree(c.ready);
    cudaFree(c.hwork);
    cudaFree(c.hsqrd);
    cudaFree(c.epart);
    cudaFree(c.counters);
    c = ChanState();
}

// antenna groups per frame for the pilot kernel: aim for about two waves of resident CTAs so that
// the GPU is filled and the tail is short (cross-CTA energy sums are combined by the last CTA of
// each frame), but keep >= 16 rows per team so the per-CTA setup (twiddles, pilot reciprocals) stays
// amortised -- unless the launch is tiny (latency configs), where every antenna gets its own team
int pilot_groups(const lsmrc_ctx* h, int n_frames)
{
    const int teams = h->ops->teams;
    const int max_g = (h->cfg.n_ant + teams - 1) / teams;
    const int min_rows = ((long long)n_frames * 4 >= h->pilot_wave) ? 16 : 1;
    int g_rows = h->cfg.n_ant / (teams * min_rows);
    if (g_rows < 1) g_rows = 1;
    int g = (2 * h->pilot_wave + n_frames - 1) / n_frames;
    if (g > g_rows) g = g_rows;
    if (g > max_g) g = max_g;
    if ((long long)g * n_frames > (long long)n_frames + kPilotCtaTarget) g = (int)(((long long)n_frames + kPilotCtaTarget) / n_frames);
    if (g < 1) g = 1;
    return g;
}

// bulk async copies of antenna rows need 16-byte aligned rows: even strides and prefix, aligned base
int rows_16b_aligned(const KernelParams& p)
{
    return (reinterpret_cast<uintptr_t>(p.rx) % 16 == 0) && p.cp % 2 == 0 && p.ant_stride % 2 == 0 && p.sym_stride % 2 == 0 &&
           p.frame_stride % 2 == 0;
}

int launch_pilot(lsmrc_ctx* h, cudaStream_t st, KernelParams p, ChanState& ch, float2* d_hconj, float* d_hsqrd)
{
    p.first_sym = 0;
    p.n_sym_work = 1;
    p.hwork = ch.hwork;
    p.hconj = d_hconj;
    p.hsqrd = d_hsqrd ? d_hsqrd : ch.hsqrd;
    p.n_groups = pilot_groups(h, p.n_frames);
    // few antennas: pack several frames into one CTA so that its teams are not idle, as long as the
    // packed grid still fills the GPU
    p.frames_per_cta = 1;
    if (p.n_groups == 1) {
        int fpc = h->ops->teams / h->cfg.n_ant;
        while (fpc > 1 && (p.n_frames + fpc - 1) / fpc < h->pilot_wave) --fpc;
        if (fpc > 1) p.frames_per_cta = fpc;
    }
    p.epart = ch.epart;
    p.counters = ch.counters;
    p.x_tma = rows_16b_aligned(p);
    {
        // tiny virtual CTAs (a round or two of row FFTs per team: few antennas, small N) amortise the per-CTA setup by
        // striding one resident wave of CTAs over them; larger ones are left to the hardware scheduler, which
        // balances them better than a static stride
        const int tpf = h->ops->teams / p.frames_per_cta;
        const int rounds = (h->cfg.n_ant + p.n_groups * tpf - 1) / (p.n_groups * tpf);
        p.pilot_grid_cap = rounds <= 2 ? h->pilot_wave : 0;
    }
    CK(h, h->ops->launch(MODE_PILOT, p, st, h->max_data_ctas));
    h->launches++;
    return LSMRC_OK;
}

int launch_data(lsmrc_ctx* h, cudaStream_t st, KernelParams p, ChanState& ch, float* d_hsqrd, int first_sym, int n_sym_work)
{
    p.first_sym = first_sym;
    p.n_sym_work = n_sym_work;
    p.hwork = ch.hwork;
    p.hsqrd = d_hsqrd ? d_hsqrd : ch.hsqrd;
    p.n_groups = 1;
    p.x_tma = rows_16b_aligned(p);
    p.ticket = ch.ticket;
    CK(h, h->ops->launch(MODE_DATA, p, st, h->max_data_ctas));
    h->launches++;
    return LSMRC_OK;
}

// Shuffle-stage plans, batches that give every team of a full wave of CTAs its own (frame, symbol) pair: pilot items, then
// data items, from one persistent launch (lsmrc_frames_sh).  Returns 1 when it launched, 0 when the kernel pair has to run.
int launch_fused(lsmrc_ctx* h, cudaStream_t st, KernelParams p, ChanState& ch, float2* d_hconj, float* d_hsqrd, cudaEvent_t ev_before)
{
    const lsmrc_config& c = h->cfg;
    if (!h->ops->launch_fused || !h->one_launch_frames || c.n_sym < 2) return 0;
    const int teams = h->ops->teams;
    const long long n_work = (long long)p.n_frames * (c.n_sym - 1);
    if ((n_work + teams - 1) / teams < (long long)h->max_data_ctas) return 0;  // (smaller batches: antenna split / wider pilot grid)
    p.n_groups = pilot_groups(h, p.n_frames);
    if (p.n_groups == 1 && teams / c.n_ant > 1) return 0;                        // (few antennas: the pilot kernel packs frames)
    p.first_sym = 1;
    p.n_sym_work = c.n_sym - 1;
    p.hwork = ch.hwork;
    p.hconj = d_hconj;
    p.hsqrd = d_hsqrd ? d_hsqrd : ch.hsqrd;
    p.frames_per_cta = 1;
    p.pilot_grid_cap = 0;
    p.epart = ch.epart;
    p.counters = ch.counters;
    p.ticket = ch.ticket;
    p.ready = ch.ready;
    p.ant_split = 1;
    p.x_tma = rows_16b_aligned(p);
    if (ev_before) CK(h, cudaEventRecord(ev_before, st));  // (no separate pilot phase: the split reported is 0 / whole)
    CK(h, h->ops->launch_fused(p, st, h->max_data_ctas));
    h->launches++;
    h->fused_calls++;
    return 1;
}

// where the symbols of ONE frame sit when they are not a dense [S][A][N+C] block (ring slots read in place)
struct RxLayout {
    long long sym_stride;  // complex elements between consecutive symbols
    bool dense = false;    // the cyclic prefix was dropped on the way in: rows of N samples, [F][S][A][N]
    const float2* rx2;     // symbols >= split_sym continue here (ring wrap); nullptr = contiguous
    int split_sym;
    int align4;            // slots are 4- but not 8-byte aligned (the reference ring's 12-byte header)
};

// pilot + data launches for n_frames whole frames (ch must hold >= n_frames); `lay` only with the
// one-launch kernel (the caller has checked that it applies)
int launch_frames(lsmrc_ctx* h, cudaStream_t st, const float2* d_rx, int n_frames, ChanState& ch, float2* d_hconj,
                  float* d_hsqrd, float2* d_comb, uint8_t* d_bits, bool timed, const RxLayout* lay = nullptr)
{
    KernelParams p = base_params(h);
    p.rx = d_rx;
    if (lay && lay->dense) {
        p.cp = 0;
        p.ant_stride = h->cfg.fft_size;
        p.sym_stride = (long long)h->cfg.n_ant * h->cfg.fft_size;
        p.frame_stride = p.sym_stride * h->cfg.n_sym;
        lay = nullptr;
    }
    if (lay) {
        p.sym_stride = lay->sym_stride;
        p.rx_align4 = lay->align4;
        if (lay->rx2) {
            p.rx2 = lay->rx2;
            p.split_sym = lay->split_sym;
        }
    }
    p.n_frames = n_frames;
    p.combined = d_comb;
    p.bits = d_bits;
    cudaEvent_t* ev = h->ev[h->ev_calls % lsmrc_ctx::kEvRing];
    if (timed) CK(h, cudaEventRecord(ev[0], st));
    const int one_as = (h->oneshot && h->one_ops && h->cfg.n_sym > 1)
                           ? h->one_ops->split(n_frames, h->cfg.n_sym - 1, h->cfg.n_ant, h->n_sms, h->smem_optin)
                           : 0;
    if (one_as > 0) {
        // launch-latency bound batch: channel estimate and data symbols in one kernel
        p.first_sym = 1;
        p.n_sym_work = h->cfg.n_sym - 1;
        p.hwork = ch.hwork;
        p.hconj = d_hconj;
        p.hsqrd = d_hsqrd ? d_hsqrd : ch.hsqrd;
        p.ant_split = one_as;
        p.twiddles = h->d_one_tw;
        if (timed) CK(h, cudaEventRecord(ev[1], st));
        CK(h, h->one_ops->launch(p, st));
        h->launches++;
        h->oneshot_calls++;
    } else {
        if (lay) return fail(h, LSMRC_ERR_STATE, "in-place ring layout without the one-launch kernel");
        int rc = launch_fused(h, st, p, ch, d_hconj, d_hsqrd, timed ? ev[1] : nullptr);
        if (rc < 0) return rc;
        if (rc == 0) {  // (1: channel estimate and data symbols of the whole batch went out as one persistent launch)
            rc = launch_pilot(h, st, p, ch, d_hconj, d_hsqrd);
            if (rc != LSMRC_OK) return rc;
            if (timed) CK(h, cudaEventRecord(ev[1], st));
            if (h->cfg.n_sym > 1) {
                rc = launch_data(h, st, p, ch, d_hsqrd, 1, h->cfg.n_sym - 1);
                if (rc != LSMRC_OK) return rc;
            }
        }
    }
    if (timed) {
        CK(h, cudaEventRecord(ev[2], st));
        h->ev_calls++;
    }
    return LSMRC_OK;
}

// largest batch the one-launch kernel processes in place in pinned host memory (beyond it PCIe bandwidth, not latency,
// decides and the staged, pipelined path is faster)
constexpr size_t kZeroCopyBytes = 512u << 10;

// device-visible alias of a pinned (page-locked, mapped) host buffer; nullptr for anything else
void* mapped_alias(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

bool is_pinned_or_device(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

struct ScopedPin {
    void* p = nullptr;
    bool pinned = false;
    void pin(const void* ptr, size_t bytes)
    {
        if (!ptr || bytes == 0 || is_pinned_or_device(ptr)) return;
        if (cudaHostRegister(const_cast<void*>(ptr), bytes, cudaHostRegisterDefault) == cudaSuccess) {
            p = const_cast<void*>(ptr);
            pinned = true;
        } else {
            cudaGetLastError();  // fall back to staged (synchronous) copies
        }
    }
    ~ScopedPin()
    {
        if (pinned) cudaHostUnregister(p);
    }
};

// whether the H2D copies of whole slots leave the cyclic prefix on the host (strided copy; rows long enough for the copy engine)
bool strip_cp_on_h2d(const lsmrc_ctx* h)
{
    const lsmrc_config& c = h->cfg;
    return h->h2d_strip_cp && c.cp_len > 0 && (size_t)c.fft_size * sizeof(float2) >= h->h2d_strip_min_row;
}

int alloc_lane(lsmrc_ctx* h, Lane& L)
{
    const lsmrc_config& c = h->cfg;
    const size_t F = (size_t)c.max_frames;
    const size_t nd = (size_t)(c.n_sym > 1 ? c.n_sym - 1 : 1);
    CK(h, cudaStreamCreateWithFlags(&L.st, cudaStreamNonBlocking));
    CK(h, cudaEventCreate(&L.copied));  // (timing enabled: the four events of a lane are the timeline of lsmrc_ring_trace)
    CK(h, cudaEventCreate(&L.done));
    CK(h, cudaEventCreate(&L.t_start));
    CK(h, cudaEventCreate(&L.t_kernels));
    CK(h, cudaMalloc(&L.d_rx, F * h->frame_elems * sizeof(float2)));
    CK(h, cudaMalloc(&L.d_hconj, F * (size_t)c.n_ant * h->K * sizeof(float2)));
    {
        const int rc = ensure_chan(h, L.ch, c.max_frames, nullptr);
        if (rc != LSMRC_OK) return rc;
    }
    CK(h, cudaMalloc(&L.d_comb, F * nd * h->K * sizeof(float2)));
    CK(h, cudaMalloc(&L.d_bits, F * nd * h->row_bytes));
    CK(h, cudaMallocHost(&L.h_comb, F * nd * h->K * sizeof(float2)));
    CK(h, cudaMallocHost(&L.h_bits, F * nd * h->row_bytes));
    CK(h, cudaMallocHost(&L.h_hconj, F * (size_t)c.n_ant * h->K * sizeof(float2)));
    return LSMRC_OK;
}

void free_lane(Lane& L)
{
    if (L.st) cudaStreamSynchronize(L.st);
    cudaFree(L.d_rx);
    cudaFree(L.d_rx16);
    cudaFree(L.d_hconj);
    free_chan(L.ch);
    cudaFree(L.d_comb);
    cudaFree(L.d_bits);
    cudaFreeHost(L.h_comb);
    cudaFreeHost(L.h_bits);
    cudaFreeHost(L.h_hconj);
    if (L.copied) cudaEventDestroy(L.copied);
    if (L.done) cudaEventDestroy(L.done);
    if (L.t_start) cudaEventDestroy(L.t_start);
    if (L.t_kernels) cudaEventDestroy(L.t_kernels);
    if (L.st) cudaStreamDestroy(L.st);
    L = Lane();
}

int ensure_lanes(lsmrc_ctx* h)
{
    if (!h->lanes.empty()) return LSMRC_OK;
    h->lanes.resize((size_t)h->cfg.n_lanes);
    for (Lane& L : h->lanes) {
        int rc = alloc_lane(h, L);
        if (rc != LSMRC_OK) {
            for (Lane& M : h->lanes) free_lane(M);
            h->lanes.clear();
            return rc;
        }
    }
    return LSMRC_OK;
}

int ensure_symbol_state(lsmrc_ctx* h)
{
    if (h->d_sym) return LSMRC_OK;
    const lsmrc_config& c = h->cfg;
    CK(h, cudaMalloc(&h->d_sym, h->slot_elems * sizeof(float2)));
    CK(h, cudaMalloc(&h->d_one_hconj, (size_t)c.n_ant * h->K * sizeof(float2)));
    {
        const int rc = ensure_chan(h, h->one_ch, 1, nullptr);
        if (rc != LSMRC_OK) return rc;
    }
    CK(h, cudaMalloc(&h->d_one_comb, (size_t)h->K * sizeof(float2)));
    CK(h, cudaMalloc(&h->d_one_bits, h->row_bytes));
    CK(h, cudaMallocHost(&h->h_one_sym, h->slot_elems * sizeof(float2)));
    CK(h, cudaMallocHost(&h->h_one_comb, (size_t)h->K * sizeof(float2)));
    CK(h, cudaMallocHost(&h->h_one_bits, h->row_bytes));
    return LSMRC_OK;
}

// stage one ring slot onto the device (the reference copies straight from pageable shm,
// ShMemSymBuff_gpu.hpp:386-387, which makes cudaMemcpyAsync synchronous)
int stage_symbol(lsmrc_ctx* h, const void* rx_sym, int on_device, const float2** d_out)
{
    if (on_device) {
        *d_out = static_cast<const float2*>(rx_sym);
        return LSMRC_OK;
    }
    const size_t bytes = h->slot_elems * sizeof(float2);
    cudaStream_t st = h->own_stream;
    const void* src = rx_sym;
    if (!is_pinned_or_device(rx_sym)) {
        CK(h, cudaStreamSynchronize(st));  // staging buffer may still be in flight
        std::memcpy(h->h_one_sym, rx_sym, bytes);
        src = h->h_one_sym;
    }
    CK(h, cudaMemcpyAsync(h->d_sym, src, bytes, cudaMemcpyHostToDevice, st));
    *d_out = h->d_sym;
    return LSMRC_OK;
}

}  // namespace

namespace {

// subcarriers per CTA of k_zf_create: kZfKT where its tile fits shared memory, else the largest power of two below that
// does (0: not even one subcarrier fits)
size_t zf_smem(int kt, int n_ant, int n_users)
{
    return sizeof(float2) * ((size_t)kt * n_ant * n_users + (size_t)kt * n_users * 2 * n_users);
}

int zf_tile(const lsmrc_ctx* h, int n_ant, int n_users)
{
    int kt = kZfKT;
    while (kt >= 1 && zf_smem(kt, n_ant, n_users) + 1024 > h->smem_optin) kt /= 2;
    return kt;
}

// The dynamic shared-memory limit of k_zf_create is a per-device, per-process attribute: lsmrc_create raises it once to the
// largest tile zf_tile can pick (smem_optin - 1024), the same value for every handle, so no handle lowers it under
// another and no call sets it (calls stay capturable).  Frames go on gridDim.y in chunks of at most 65535.
// ginv_diag (may be nullptr): [F][U][K] diagonal of inv(G), frame stride U * K.
int launch_zf_create(lsmrc_ctx* h, cudaStream_t st, const float2* x, float2* hzf, int n_ant, int n_sc, int n_users, int kt, float lambda,
                     int n_frames, long long x_frame_stride, long long x_user_stride, long long hzf_frame_stride, int* d_count,
                     float* ginv_diag = nullptr)
{
    const size_t smem = zf_smem(kt, n_ant, n_users);
    constexpr int kMaxGridY = 65535;
    for (int f0 = 0; f0 < n_frames; f0 += kMaxGridY) {
        const int nf = n_frames - f0 < kMaxGridY ? n_frames - f0 : kMaxGridY;
        const dim3 grid((unsigned)((n_sc + kt - 1) / kt), (unsigned)nf);
        k_zf_create<<<grid, 128, smem, st>>>(x + f0 * x_frame_stride, hzf + f0 * hzf_frame_stride, n_ant, n_sc, n_users, kt, lambda,
                                             x_frame_stride, x_user_stride, hzf_frame_stride, d_count,
                                             ginv_diag ? ginv_diag + (long long)f0 * n_users * n_sc : nullptr);
        h->launches++;
        CK(h, cudaGetLastError());
    }
    return LSMRC_OK;
}

// device scratch that only grows (a call after one of the same size allocates nothing: CUDA-graph capturable)
template <class T>
int ensure_scratch(lsmrc_ctx* h, T*& ptr, size_t& cap, size_t bytes, cudaStream_t quiesce)
{
    if (cap >= bytes) return LSMRC_OK;
    CK(h, cudaStreamSynchronize(quiesce));
    cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    CK(h, cudaMalloc(&ptr, bytes));
    cap = bytes;
    return LSMRC_OK;
}

// a plan's twiddle table (twn entries, written by fill) into a new device buffer
int upload_twiddles(lsmrc_ctx* h, void (*fill)(float2*), int twn, float2** d_tw)
{
    std::vector<float2> tw((size_t)twn);
    fill(tw.data());
    cudaError_t e;
    if ((e = cudaMalloc(d_tw, tw.size() * sizeof(float2))) != cudaSuccess) return fail_cuda(h, e, "cudaMalloc twiddles");
    if ((e = cudaMemcpy(*d_tw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice)) != cudaSuccess) return fail_cuda(h, e, "cudaMemcpy twiddles");
    return LSMRC_OK;
}

}  // namespace

extern "C" {

int lsmrc_abi_version(void) { return LSMRC_ABI_VERSION; }

const char* lsmrc_error_name(int code)
{
    switch (code) {
        case LSMRC_OK: return "LSMRC_OK";
        case LSMRC_ERR_INVALID: return "LSMRC_ERR_INVALID";
        case LSMRC_ERR_CUDA: return "LSMRC_ERR_CUDA";
        case LSMRC_ERR_UNSUPPORTED: return "LSMRC_ERR_UNSUPPORTED";
        case LSMRC_ERR_NO_PILOT: return "LSMRC_ERR_NO_PILOT";
        case LSMRC_ERR_NO_DEVICE: return "LSMRC_ERR_NO_DEVICE";
        case LSMRC_ERR_STATE: return "LSMRC_ERR_STATE";
        default: return "LSMRC_ERR_UNKNOWN";
    }
}

const char* lsmrc_last_error(lsmrc_handle h)
{
    if (h) return h->err.c_str();
    std::lock_guard<std::mutex> g(g_err_mutex);
    static thread_local std::string copy;
    copy = g_create_error;
    return copy.c_str();
}

size_t lsmrc_bits_row_bytes(int fft_size, int qam_bits)
{
    if (fft_size < 2 || qam_bits < 1) return 0;
    return ((size_t)(fft_size - 1) * (size_t)qam_bits + 7u) / 8u;
}

size_t lsmrc_rx_frame_elems(const lsmrc_config* c)
{
    if (!c) return 0;
    return (size_t)c->n_sym * (size_t)c->n_ant * (size_t)(c->fft_size + c->cp_len);
}

int lsmrc_supported_fft_size(int fft_size) { return find_plan(fft_size) != nullptr; }

int lsmrc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int lsmrc_device_pci_bus_id(int device, char* buf, size_t buf_len)
{
    if (!buf || buf_len < 13) return LSMRC_ERR_INVALID;
    if (cudaDeviceGetPCIBusId(buf, (int)buf_len, device) != cudaSuccess) {
        cudaGetLastError();
        return LSMRC_ERR_CUDA;
    }
    return LSMRC_OK;
}

int lsmrc_create(const lsmrc_config* cfg, lsmrc_handle* out)
{
    if (!cfg || !out) return fail(nullptr, LSMRC_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->n_ant < 1 || cfg->n_sym < 1 || cfg->cp_len < 0 || cfg->max_frames < 1 || cfg->n_lanes < 1 ||
        cfg->n_lanes > 64)
        return fail(nullptr, LSMRC_ERR_INVALID, "n_ant/n_sym/max_frames/n_lanes must be >= 1, cp_len >= 0");
    if (cfg->qam_bits != 2 && cfg->qam_bits != 4 && cfg->qam_bits != 6)
        return fail(nullptr, LSMRC_ERR_UNSUPPORTED, "qam_bits must be 2, 4 or 6");
    const PlanOps* ops = find_plan(cfg->fft_size);
    if (!ops) return fail(nullptr, LSMRC_ERR_UNSUPPORTED, "fft_size must be a power of two in 64..4096");

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, LSMRC_ERR_NO_DEVICE,
                    std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, LSMRC_ERR_INVALID, "device ordinal out of range");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) return fail_cuda(nullptr, e, "cudaGetDeviceProperties");
    if (prop.major != 10)
        return fail(nullptr, LSMRC_ERR_NO_DEVICE,
                    std::string("device is ") + prop.name + " (sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                        "); this library is built for sm_100a only");
    if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) return fail_cuda(nullptr, e, "cudaSetDevice");

    lsmrc_ctx* h = new lsmrc_ctx();
    h->cfg = *cfg;
    h->K = cfg->fft_size - 1;
    h->row_bytes = lsmrc_bits_row_bytes(cfg->fft_size, cfg->qam_bits);
    h->slot_elems = (size_t)cfg->n_ant * (size_t)(cfg->fft_size + cfg->cp_len);
    h->frame_elems = (size_t)cfg->n_sym * h->slot_elems;
    h->ops = ops;

    auto bail = [&](int rc) {
        std::string msg = h->err;
        lsmrc_destroy(h);
        return fail(nullptr, rc, msg);
    };
    {
        int per_sm = 0, pilot_per_sm = 0;
        if ((e = ops->prepare(&per_sm, &pilot_per_sm)) != cudaSuccess) { fail_cuda(h, e, "cudaFuncSetAttribute"); return bail(LSMRC_ERR_CUDA); }
        if (per_sm < 1 || pilot_per_sm < 1) { h->err = "kernel does not fit on an SM"; return bail(LSMRC_ERR_CUDA); }
        h->max_data_ctas = per_sm * prop.multiProcessorCount;
        h->pilot_wave = pilot_per_sm * prop.multiProcessorCount;
        h->n_sms = prop.multiProcessorCount;
        h->smem_optin = prop.sharedMemPerBlockOptin;
    }
    if ((e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) { fail_cuda(h, e, "cudaStreamCreate"); return bail(LSMRC_ERR_CUDA); }
    for (int i = 0; i < lsmrc_ctx::kEvRing; ++i)
        for (int j = 0; j < 3; ++j)
            if ((e = cudaEventCreate(&h->ev[i][j])) != cudaSuccess) { fail_cuda(h, e, "cudaEventCreate"); return bail(LSMRC_ERR_CUDA); }
    if (upload_twiddles(h, ops->fill_twiddles, ops->twn, &h->d_tw) != LSMRC_OK) return bail(LSMRC_ERR_CUDA);
    if (const char* ev = std::getenv("LSMRC_H2D_STRIP_MIN_ROW")) {  // tuning/A-B knob
        const long v = std::atol(ev);
        h->h2d_strip_cp = v > 0;
        if (v > 0) h->h2d_strip_min_row = (size_t)v;
    }
    if ((h->one_ops = find_oneshot_plan(cfg->fft_size)) != nullptr) {
        const OneshotOps* oo = h->one_ops;
        if ((e = oo->prepare((int)prop.sharedMemPerBlockOptin)) != cudaSuccess) { fail_cuda(h, e, "cudaFuncSetAttribute (one-launch kernel)"); return bail(LSMRC_ERR_CUDA); }
        if (upload_twiddles(h, oo->fill_twiddles, oo->twn, &h->d_one_tw) != LSMRC_OK) return bail(LSMRC_ERR_CUDA);
    }
    if ((e = cudaMalloc(&h->d_pilot_bin, (size_t)h->K * sizeof(float2))) != cudaSuccess) { fail_cuda(h, e, "cudaMalloc pilot"); return bail(LSMRC_ERR_CUDA); }
    // zero forcing: allow the largest tile once (see launch_zf_create)
    if ((e = cudaFuncSetAttribute(k_zf_create, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(h->smem_optin - 1024))) != cudaSuccess) {
        fail_cuda(h, e, "cudaFuncSetAttribute (zero forcing)");
        return bail(LSMRC_ERR_CUDA);
    }
    {  // downlink precode kernel: its shared-memory attribute once here, so that no call sets one (calls stay capturable)
        int per_sm = 0;
        if ((e = ops->dl_prepare(&per_sm)) != cudaSuccess) { fail_cuda(h, e, "cudaFuncSetAttribute (precode kernel)"); return bail(LSMRC_ERR_CUDA); }
        if (per_sm < 1) { h->err = "precode kernel does not fit on an SM"; return bail(LSMRC_ERR_CUDA); }
        h->dl_max_ctas = per_sm * h->n_sms;
    }
    // the table uploads above are pageable-memory copies on the legacy stream (they return once staged); the kernels
    // run on non-blocking streams that do not order against it
    if ((e = cudaDeviceSynchronize()) != cudaSuccess) { fail_cuda(h, e, "cudaDeviceSynchronize"); return bail(LSMRC_ERR_CUDA); }
    *out = h;
    return LSMRC_OK;
}

int lsmrc_destroy(lsmrc_handle h)
{
    if (!h) return LSMRC_ERR_INVALID;
    cudaSetDevice(h->cfg.device);
    if (h->own_stream) cudaStreamSynchronize(h->own_stream);
    for (Lane& L : h->lanes) free_lane(L);
    cudaFree(h->d_tw);
    cudaFree(h->d_one_tw);
    cudaFree(h->d_noise_part);
    cudaFree(h->d_hit);
    cudaFree(h->d_pilot_bin);
    free_chan(h->dev_ch);
    free_chan(h->one_ch);
    free_chan(h->mu_ch);
    cudaFree(h->d_mu_hconj);
    cudaFree(h->d_mu_ls);
    cudaFree(h->d_mu_hzf);
    cudaFree(h->d_mu_wd);
    cudaFree(h->d_mu_soft);
    cudaFree(h->d_mu_count);
    cudaFree(h->d_dl_hzf);
    cudaFree(h->d_dl_pd);
    cudaFree(h->d_dl_part);
    cudaFree(h->d_sym);
    cudaFree(h->d_one_hconj);
    cudaFree(h->d_one_comb);
    cudaFree(h->d_one_bits);
    cudaFreeHost(h->h_one_sym);
    cudaFreeHost(h->h_one_comb);
    cudaFreeHost(h->h_one_bits);
    for (int i = 0; i < lsmrc_ctx::kEvRing; ++i)
        for (int j = 0; j < 3; ++j)
            if (h->ev[i][j]) cudaEventDestroy(h->ev[i][j]);
    if (h->ring_epoch) cudaEventDestroy(h->ring_epoch);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    cudaGetLastError();
    delete h;
    return LSMRC_OK;
}

int lsmrc_set_pilot(lsmrc_handle h, const float* pilot_asc, int K)
{
    if (!h || !pilot_asc) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (K != h->K) return fail(h, LSMRC_ERR_INVALID, "pilot length must be fft_size-1");
    CK(h, cudaSetDevice(h->cfg.device));
    // Pilots.dat is ascending frequency; the kernels index by FFT bin.  Same roll as
    // matrix_readX (cpuLS.hpp:105-112): X_bin[k] = P[(k + (K+1)/2) mod K].
    std::vector<float2> xb((size_t)K);
    const float2* P = reinterpret_cast<const float2*>(pilot_asc);
    for (int k = 0; k < K; ++k) {
        xb[(size_t)k] = P[(k + (K + 1) / 2) % K];
        if (xb[(size_t)k].x == 0.f && xb[(size_t)k].y == 0.f) return fail(h, LSMRC_ERR_INVALID, "pilot contains a zero subcarrier");
    }
    // no kernel of this handle may still be reading the old pilot, and the new one must have landed before the
    // next launch on any of the handle's (non-blocking) streams
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(h->d_pilot_bin, xb.data(), (size_t)K * sizeof(float2), cudaMemcpyHostToDevice));
    CK(h, cudaDeviceSynchronize());
    h->have_pilot = true;
    return LSMRC_OK;
}

int lsmrc_set_pilot_file(lsmrc_handle h, const char* path)
{
    if (!h) return LSMRC_ERR_INVALID;
    std::vector<float2> p((size_t)h->K);
    int used_fallback = 0;
    FILE* f = path ? std::fopen(path, "rb") : nullptr;
    if (!f) {
        // CPU-reference fallback (cpuLS.hpp:85-88).  The GPU reference uses 1+1i instead
        // (gpuLS.cu:58-62); the two disagree, we follow the CPU path we are checked against.
        for (float2& v : p) v = make_float2(0.707f, 0.707f);
        used_fallback = 1;
    } else {
        const size_t got = std::fread(p.data(), sizeof(float2), p.size(), f);
        std::fclose(f);
        if (got != p.size()) return fail(h, LSMRC_ERR_INVALID, "pilot file shorter than K complex64 values");
    }
    const int rc = lsmrc_set_pilot(h, reinterpret_cast<const float*>(p.data()), h->K);
    return rc == LSMRC_OK ? used_fallback : rc;
}

int lsmrc_demod_frames_device(lsmrc_handle h, const void* d_rx, int n_frames, void* d_hconj, void* d_hsqrd,
                              void* d_combined, void* d_bits)
{
    if (!h || !d_rx || !d_combined) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    if (n_frames == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    {
        const int rc = ensure_chan(h, h->dev_ch, n_frames, compute_stream(h));
        if (rc != LSMRC_OK) return rc;
    }
    return launch_frames(h, compute_stream(h), static_cast<const float2*>(d_rx), n_frames, h->dev_ch,
                         static_cast<float2*>(d_hconj), static_cast<float*>(d_hsqrd), static_cast<float2*>(d_combined),
                         static_cast<uint8_t*>(d_bits), h->timing);
}

}  // extern "C"

namespace {

// The multi-user calls (lsmrc_demod_frames_device_mu and _mu_soft) share their argument checks (mu_check), phases 1-2
// (mu_detect: scratch, per-user LS channel, detector build) and the hand-back (mu_finish); they differ in phase 3.
// Both read the handle's pilot layout (h->mu_pilots) when they enqueue: a captured graph keeps the one it saw.
int mu_check(lsmrc_ctx* h, const void* d_rx, const void* d_combined, int n_frames, int n_users, int detector, float noise_var)
{
    if (!h || !d_rx || !d_combined) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    const int A = h->cfg.n_ant, S = h->cfg.n_sym;
    if (h->mu_pilots == LSMRC_MU_PILOTS_COMB) {
        if (n_users < 1 || n_users > kZfMaxUsers || n_users > A || S < 2)
            return fail(h, LSMRC_ERR_INVALID, "comb pilots need 1 <= n_users <= 16, n_users <= n_ant and n_sym >= 2");
    } else if (n_users < 1 || n_users > kZfMaxUsers || n_users > A || n_users >= S) {
        return fail(h, LSMRC_ERR_INVALID, "need 1 <= n_users <= 16, n_users <= n_ant and n_users < n_sym");
    }
    if (detector != LSMRC_DETECT_ZF && detector != LSMRC_DETECT_MMSE) return fail(h, LSMRC_ERR_INVALID, "unknown detector");
    if (detector == LSMRC_DETECT_MMSE && !(std::isfinite(noise_var) && noise_var > 0.f))
        return fail(h, LSMRC_ERR_INVALID, "MMSE needs a finite noise_var > 0");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    return LSMRC_OK;
}

// Phases 1-2 on stream st for n_frames >= 1.  Wd is sized for the plan's users per pass of the data kernel (mu_ug);
// with `soft`, ginv_diag receives inv(G)'s diagonal [F][U][K].  On return p holds the data kernel's parameters except
// its outputs.
int mu_detect(lsmrc_ctx* h, cudaStream_t st, const void* d_rx, int n_frames, int n_users, int detector, float noise_var, bool count,
              bool soft, KernelParams& p)
{
    const int A = h->cfg.n_ant, S = h->cfg.n_sym, N = h->cfg.fft_size, K = h->K;
    const int kt = zf_tile(h, A, n_users);
    if (kt < 1) return fail(h, LSMRC_ERR_UNSUPPORTED, "n_ant * n_users too large for one CTA's shared memory");
    const int U = n_users, UG = h->ops->mu_ug, UP = (U + UG - 1) / UG * UG;
    const long long F = n_frames;
    int rc;
    if ((rc = ensure_chan(h, h->mu_ch, n_frames, st)) != LSMRC_OK) return rc;
    const bool comb = h->mu_pilots == LSMRC_MU_PILOTS_COMB;
    if ((rc = ensure_scratch(h, h->d_mu_hconj, h->mu_hconj_cap, sizeof(float2) * (size_t)(U * F * A * K), st)) != LSMRC_OK) return rc;
    if (comb && (rc = ensure_scratch(h, h->d_mu_ls, h->mu_ls_cap, sizeof(float2) * (size_t)(F * A * K), st)) != LSMRC_OK) return rc;
    if ((rc = ensure_scratch(h, h->d_mu_hzf, h->mu_hzf_cap, sizeof(float2) * (size_t)(F * K * U * A), st)) != LSMRC_OK) return rc;
    if ((rc = ensure_scratch(h, h->d_mu_wd, h->mu_wd_cap, sizeof(float2) * (size_t)(F * UP * A * N), st)) != LSMRC_OK) return rc;
    if (soft && (rc = ensure_scratch(h, h->d_mu_soft, h->mu_soft_cap, (sizeof(float2) + sizeof(float)) * (size_t)(F * U * K), st)) != LSMRC_OK)
        return rc;
    if (!h->d_mu_count) CK(h, cudaMalloc(&h->d_mu_count, sizeof(int)));
    int& max_ctas = soft ? h->mu_soft_max_ctas : h->mu_max_ctas;
    if (max_ctas == 0) {
        int per_sm = 0;
        CK(h, h->ops->mu_prepare(soft, &per_sm));
        if (per_sm < 1) return fail(h, LSMRC_ERR_CUDA, "multi-user data kernel does not fit on an SM");
        max_ctas = per_sm * h->n_sms;
    }
    // 1. LS channel of every user: the single-user pilot launch, once per pilot symbol (time-orthogonal pilots), or
    //    once on the comb symbol 0 followed by each user's interpolation across its own subcarriers (comb pilots)
    p = base_params(h);
    p.n_frames = n_frames;
    const long long user_elems = F * A * K;
    const int n_pilot_sym = comb ? 1 : U;
    if (comb) {
        p.rx = static_cast<const float2*>(d_rx);
        if ((rc = launch_pilot(h, st, p, h->mu_ch, h->d_mu_ls, nullptr)) != LSMRC_OK) return rc;
        const long long rows = F * A, cap = (long long)h->n_sms * 16;
        k_mu_comb_interp<<<(unsigned)(rows < cap ? rows : cap), 256, sizeof(float2) * (size_t)K, st>>>(h->d_mu_ls, h->d_mu_hconj, N, U,
                                                                                                      rows, user_elems);
        h->launches++;
        CK(h, cudaGetLastError());
    } else {
        for (int u = 0; u < U; ++u) {
            p.rx = static_cast<const float2*>(d_rx) + (long long)u * p.sym_stride;
            if ((rc = launch_pilot(h, st, p, h->mu_ch, h->d_mu_hconj + u * user_elems, nullptr)) != LSMRC_OK) return rc;
        }
    }
    // 2. detector per (frame, subcarrier): X = conj(H) [U][A][K] of the frame -> Hzf = conj(W)
    if (count) CK(h, cudaMemsetAsync(h->d_mu_count, 0, sizeof(int), st));
    if ((rc = launch_zf_create(h, st, h->d_mu_hconj, h->d_mu_hzf, A, K, U, kt, detector == LSMRC_DETECT_MMSE ? noise_var : 0.f, n_frames,
                               (long long)A * K, user_elems, (long long)K * U * A, count ? h->d_mu_count : nullptr,
                               soft ? h->d_mu_soft + 2 * F * U * K : nullptr)) != LSMRC_OK)
        return rc;
    p.rx = static_cast<const float2*>(d_rx);
    p.first_sym = n_pilot_sym;
    p.n_sym_work = S - n_pilot_sym;
    return LSMRC_OK;
}

// after phase 3: conj(H) to the caller's layout, the singular count back to the host
int mu_finish(lsmrc_ctx* h, cudaStream_t st, int n_frames, int n_users, void* d_hconj, int* n_singular)
{
    const int A = h->cfg.n_ant, K = h->K, U = n_users;
    const long long user_elems = (long long)n_frames * A * K;
    if (d_hconj) {  // [U][F][A][K] -> [F][U][A][K]
        const size_t row = sizeof(float2) * (size_t)A * K;
        for (int u = 0; u < U; ++u)
            CK(h, cudaMemcpy2DAsync(static_cast<float2*>(d_hconj) + (size_t)u * A * K, row * U, h->d_mu_hconj + u * user_elems, row, row,
                                    (size_t)n_frames, cudaMemcpyDeviceToDevice, st));
    }
    if (n_singular) {
        CK(h, cudaMemcpyAsync(n_singular, h->d_mu_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(h, cudaStreamSynchronize(st));
    }
    return LSMRC_OK;
}

}  // namespace

extern "C" {

int lsmrc_demod_frames_device_mu(lsmrc_handle h, const void* d_rx, int n_frames, int n_users, int detector, float noise_var,
                                 void* d_hconj, void* d_combined, void* d_bits, int* n_singular)
{
    int rc;
    if ((rc = mu_check(h, d_rx, d_combined, n_frames, n_users, detector, noise_var)) != LSMRC_OK) return rc;
    if (n_frames == 0) {
        if (n_singular) *n_singular = 0;
        return LSMRC_OK;
    }
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    KernelParams p;
    if ((rc = mu_detect(h, st, d_rx, n_frames, n_users, detector, noise_var, n_singular != nullptr, false, p)) != LSMRC_OK)
        return rc;
    // 3. detection fused with the row FFT of every data symbol
    p.combined = static_cast<float2*>(d_combined);
    p.bits = static_cast<uint8_t*>(d_bits);
    CK(h, h->ops->mu_launch(false, p, h->d_mu_hzf, h->d_mu_wd, nullptr, n_users, h->mu_max_ctas, h->n_sms, st));
    h->launches += 2;
    return mu_finish(h, st, n_frames, n_users, d_hconj, n_singular);
}

int lsmrc_demod_frames_device_mu_soft(lsmrc_handle h, const void* d_rx, int n_frames, int n_users, int detector, float noise_var,
                                      void* d_hconj, void* d_combined, void* d_bits, void* d_llr, void* d_sinr, int* n_singular)
{
    if (!d_llr) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (!(std::isfinite(noise_var) && noise_var > 0.f)) return fail(h, LSMRC_ERR_INVALID, "soft output needs a finite noise_var > 0");
    int rc;
    if ((rc = mu_check(h, d_rx, d_combined, n_frames, n_users, detector, noise_var)) != LSMRC_OK) return rc;
    if (n_frames == 0) {
        if (n_singular) *n_singular = 0;
        return LSMRC_OK;
    }
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    KernelParams p;
    if ((rc = mu_detect(h, st, d_rx, n_frames, n_users, detector, noise_var, n_singular != nullptr, true, p)) != LSMRC_OK)
        return rc;
    // 3a. (rho, scale) per (frame, user, subcarrier) from the diagonal of inv(G)
    const long long n = (long long)n_frames * n_users * h->K;
    float2* tab = reinterpret_cast<float2*>(h->d_mu_soft);
    long long blocks = (n + 255) / 256;
    if (blocks > (long long)h->n_sms * 16) blocks = (long long)h->n_sms * 16;
    k_mu_soft_scale<<<(unsigned)blocks, 256, 0, st>>>(h->d_mu_soft + 2 * n, tab, static_cast<float*>(d_sinr), n, h->K,
                                                      detector == LSMRC_DETECT_MMSE ? 1 : 0, noise_var, noise_var);
    h->launches++;
    CK(h, cudaGetLastError());
    // 3b. detection fused with the row FFT, with the soft epilogue
    p.combined = static_cast<float2*>(d_combined);
    p.bits = static_cast<uint8_t*>(d_bits);
    p.llr = static_cast<float*>(d_llr);
    CK(h, h->ops->mu_launch(true, p, h->d_mu_hzf, h->d_mu_wd, tab, n_users, h->mu_soft_max_ctas, h->n_sms, st));
    h->launches += 2;
    return mu_finish(h, st, n_frames, n_users, d_hconj, n_singular);
}

int lsmrc_precode_frames_device(lsmrc_handle h, const void* d_hconj, int n_frames, int n_users, float reg, const void* d_sym,
                                int n_sym_dl, void* d_tx, void* d_gain, int* n_singular)
{
    if (!h || !d_hconj || !d_sym || !d_tx) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    const int A = h->cfg.n_ant, N = h->cfg.fft_size, C = h->cfg.cp_len, K = h->K, U = n_users;
    if (U < 1 || U > kZfMaxUsers || U > A) return fail(h, LSMRC_ERR_INVALID, "need 1 <= n_users <= 16 and n_users <= n_ant");
    if (n_sym_dl < 1) return fail(h, LSMRC_ERR_INVALID, "n_sym_dl must be >= 1");
    if (!(std::isfinite(reg) && reg >= 0.f)) return fail(h, LSMRC_ERR_INVALID, "reg must be finite and >= 0");
    if (C > N) return fail(h, LSMRC_ERR_INVALID, "a cyclic prefix longer than the symbol cannot be transmitted");
    const int kt = zf_tile(h, A, U);
    if (kt < 1) return fail(h, LSMRC_ERR_UNSUPPORTED, "n_ant * n_users too large for one CTA's shared memory");
    if (n_frames == 0) {
        if (n_singular) *n_singular = 0;
        return LSMRC_OK;
    }
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    const long long F = n_frames;
    const long long frame_elems = (long long)K * U * A;  // one frame's precoder block
    constexpr int kChunk = 4096;                         // elements per power partial
    const int n_chunks = (int)((frame_elems + kChunk - 1) / kChunk);
    int rc;
    if ((rc = ensure_scratch(h, h->d_dl_hzf, h->dl_hzf_cap, sizeof(float2) * (size_t)(F * frame_elems), st)) != LSMRC_OK) return rc;
    if ((rc = ensure_scratch(h, h->d_dl_pd, h->dl_pd_cap, sizeof(float2) * (size_t)(F * U * A * N), st)) != LSMRC_OK) return rc;
    if ((rc = ensure_scratch(h, h->d_dl_part, h->dl_part_cap, sizeof(float) * (size_t)(F * n_chunks + F), st)) != LSMRC_OK) return rc;
    if (!h->d_mu_count) CK(h, cudaMalloc(&h->d_mu_count, sizeof(int)));
    // lsmrc_set_timing: the two phases on the handle's event ring (lsmrc_last_kernel_ms: precoder build, precode)
    cudaEvent_t* ev = h->timing ? h->ev[h->ev_calls % lsmrc_ctx::kEvRing] : nullptr;
    if (ev) CK(h, cudaEventRecord(ev[0], st));
    // 1. precoder per (frame, subcarrier): X = conj(H) [U][A][K] of the frame, as the caller has it -> Hzf = conj(P)
    if (n_singular) CK(h, cudaMemsetAsync(h->d_mu_count, 0, sizeof(int), st));
    if ((rc = launch_zf_create(h, st, static_cast<const float2*>(d_hconj), h->d_dl_hzf, A, K, U, kt, reg, n_frames, frame_elems,
                               (long long)A * K, frame_elems, n_singular ? h->d_mu_count : nullptr)) != LSMRC_OK)
        return rc;
    // 2. per-frame gain from the sum of |P|^2 in a fixed order
    float* gain = d_gain ? static_cast<float*>(d_gain) : h->d_dl_part + F * n_chunks;
    k_sq_norm_chunks<<<(unsigned)(F * n_chunks), 256, 0, st>>>(h->d_dl_hzf, frame_elems, kChunk, n_chunks, h->d_dl_part);
    k_dl_gain<<<(unsigned)((F + 7) / 8), 256, 0, st>>>(h->d_dl_part, n_chunks, n_frames, (float)U * (float)K, gain);
    h->launches += 2;
    CK(h, cudaGetLastError());
    if (ev) CK(h, cudaEventRecord(ev[1], st));
    // 3. bin-order precoder, then precoding fused with the inverse row FFT and the cyclic prefix
    CK(h, h->ops->dl_launch(h->d_dl_hzf, h->d_dl_pd, static_cast<const float2*>(d_sym), gain, static_cast<float2*>(d_tx), h->d_tw,
                            n_frames, n_sym_dl, A, U, C, h->dl_max_ctas, h->n_sms, st));
    h->launches += 2;
    if (ev) {
        CK(h, cudaEventRecord(ev[2], st));
        h->ev_calls++;
    }
    if (n_singular) {
        CK(h, cudaMemcpyAsync(n_singular, h->d_mu_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(h, cudaStreamSynchronize(st));
    }
    return LSMRC_OK;
}

int lsmrc_demod_frames_device_soft(lsmrc_handle h, const void* d_rx, int n_frames, void* d_combined, void* d_bits,
                                   void* d_llr, float noise_var)
{
    if (!h || !d_rx || !d_combined || !d_llr) return fail(h, LSMRC_ERR_INVALID, "null argument");
    // the epilogue scales by 1/noise_var: +inf, and subnormals whose reciprocal overflows, would give +-inf or NaN LLRs
    if (!(std::isfinite(noise_var) && noise_var > 0.f && std::isfinite(1.0f / noise_var)))
        return fail(h, LSMRC_ERR_INVALID, "soft output needs a finite noise_var > 0 with a finite reciprocal");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    if (n_frames == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    {
        const int rc = ensure_chan(h, h->dev_ch, n_frames, compute_stream(h));
        if (rc != LSMRC_OK) return rc;
    }
    h->soft_llr = static_cast<float*>(d_llr);
    h->soft_inv_noise = 1.0f / noise_var;
    const int rc = launch_frames(h, compute_stream(h), static_cast<const float2*>(d_rx), n_frames, h->dev_ch, nullptr, nullptr,
                                 static_cast<float2*>(d_combined), static_cast<uint8_t*>(d_bits), h->timing);
    h->soft_llr = nullptr;
    return rc;
}

int lsmrc_estimate_noise_var(lsmrc_handle h, const void* d_combined, const void* d_hsqrd, int n_frames, void* d_noise_var)
{
    if (!h || !d_combined || !d_hsqrd || !d_noise_var) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    const int nd = h->cfg.n_sym - 1;
    if (nd < 1) return fail(h, LSMRC_ERR_STATE, "no data symbols in a frame");
    if (n_frames == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    const size_t rows = (size_t)n_frames * nd;
    if (rows > h->noise_part_rows) {
        CK(h, cudaStreamSynchronize(st));
        cudaFree(h->d_noise_part);
        h->d_noise_part = nullptr;
        h->noise_part_rows = 0;
        CK(h, cudaMalloc(&h->d_noise_part, rows * sizeof(float)));
        h->noise_part_rows = rows;
    }
    k_noise_rows<<<(unsigned)rows, 256, 0, st>>>(static_cast<const float2*>(d_combined), static_cast<const float*>(d_hsqrd), h->K, nd,
                                                 h->cfg.qam_bits, h->d_noise_part);
    k_noise_frames<<<(unsigned)((n_frames + 7) / 8), 256, 0, st>>>(h->d_noise_part, nd, h->K, n_frames, static_cast<float*>(d_noise_var));
    h->launches += 2;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_llr_from_combined(lsmrc_handle h, const void* d_combined, const void* d_hsqrd, const void* d_noise_var, int n_frames,
                            void* d_llr)
{
    if (!h || !d_combined || !d_hsqrd || !d_noise_var || !d_llr) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    const int nd = h->cfg.n_sym - 1;
    if (nd < 1) return fail(h, LSMRC_ERR_STATE, "no data symbols in a frame");
    if (n_frames == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    const long long n_sym = (long long)n_frames * nd * h->K;
    const float2* y = static_cast<const float2*>(d_combined);
    const float* e = static_cast<const float*>(d_hsqrd);
    const float* nv = static_cast<const float*>(d_noise_var);
    float* out = static_cast<float*>(d_llr);
    long long blocks = (n_sym + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    const unsigned g = (unsigned)blocks;
    if (h->cfg.qam_bits == 2) k_llr_rows<2><<<g, 256, 0, st>>>(y, e, nv, h->K, nd, n_sym, out);
    else if (h->cfg.qam_bits == 4) k_llr_rows<4><<<g, 256, 0, st>>>(y, e, nv, h->K, nd, n_sym, out);
    else k_llr_rows<6><<<g, 256, 0, st>>>(y, e, nv, h->K, nd, n_sym, out);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_zf_create(lsmrc_handle h, const void* d_x, int n_ant, int n_sc, int n_users, void* d_hzf, int* n_singular)
{
    if (!h || !d_x || !d_hzf) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_ant < 1 || n_sc < 1 || n_users < 1 || n_users > kZfMaxUsers) return fail(h, LSMRC_ERR_INVALID, "need n_ant, n_sc >= 1 and 1 <= n_users <= 16");
    if (n_users > n_ant) return fail(h, LSMRC_ERR_INVALID, "more users than antennas: X X^H would be singular");
    const int kt = zf_tile(h, n_ant, n_users);
    if (kt < 1) return fail(h, LSMRC_ERR_UNSUPPORTED, "n_ant * n_users too large for one CTA's shared memory");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    if (!h->d_hit) CK(h, cudaMalloc(&h->d_hit, sizeof(unsigned long long)));
    int* d_count = reinterpret_cast<int*>(h->d_hit);
    CK(h, cudaMemsetAsync(d_count, 0, sizeof(int), st));
    {
        const int rc = launch_zf_create(h, st, static_cast<const float2*>(d_x), static_cast<float2*>(d_hzf), n_ant, n_sc, n_users, kt, 0.f, 1,
                                        0, (long long)n_ant * n_sc, 0, d_count);
        if (rc != LSMRC_OK) return rc;
    }
    if (n_singular) {
        CK(h, cudaMemcpyAsync(n_singular, d_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(h, cudaStreamSynchronize(st));
    }
    return LSMRC_OK;
}

int lsmrc_zf_apply(lsmrc_handle h, const void* d_hzf, const void* d_xd, int n_ant, int n_sc, int n_users, void* d_hx)
{
    if (!h || !d_hzf || !d_xd || !d_hx) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_ant < 1 || n_sc < 1 || n_users < 1) return fail(h, LSMRC_ERR_INVALID, "bad dimensions");
    CK(h, cudaSetDevice(h->cfg.device));
    long long blocks = ((long long)n_ant * n_sc + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_zf_apply<<<(unsigned)blocks, 256, 0, compute_stream(h)>>>(static_cast<const float2*>(d_hzf), static_cast<const float2*>(d_xd),
                                                               static_cast<float2*>(d_hx), n_ant, n_sc, n_users);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

// wire-format samples to complex float: out[r][n] = float(in[r][skip + n]) * scale (k_sc16_to_fc32)
static int launch_sc16_to_fc32(lsmrc_ctx* h, cudaStream_t st, float2* out, const short2* in, long long rows, int n_in, int skip, int n_out,
                               float scale)
{
    const bool vec2 = ((n_in | skip | n_out) & 1) == 0 && reinterpret_cast<uintptr_t>(in) % 8 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
    long long blocks = (rows * (n_out / (vec2 ? 2 : 1)) + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    if (vec2)
        k_sc16_to_fc32<true><<<(unsigned)blocks, 256, 0, st>>>(out, in, rows, n_in, skip, n_out, scale);
    else
        k_sc16_to_fc32<false><<<(unsigned)blocks, 256, 0, st>>>(out, in, rows, n_in, skip, n_out, scale);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

// sc16: h_rx holds the radio's wire format (int16 I/Q, 4 bytes per sample), converted on the device after the copy
static int demod_frames_host_impl(lsmrc_handle h, const void* h_rx, int n_frames, void* h_hconj, void* h_hsqrd, void* h_combined,
                                  void* h_bits, bool sc16, float scale)
{
    if (!h || !h_rx || !h_combined) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(h, LSMRC_ERR_INVALID, "n_frames < 0");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    if (n_frames == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    const lsmrc_config& c = h->cfg;
    const size_t nd = (size_t)(c.n_sym - 1);
    const size_t elem = sc16 ? sizeof(short2) : sizeof(float2);  // bytes per sample on the host
    const size_t rx_fb = h->frame_elems * elem;
    // Latency path: a batch the one-launch kernel takes, in pinned host memory and small enough that
    // PCIe latency rather than bandwidth decides, is processed in place -- the kernel loads the
    // antenna-samples from and stores the results to the host buffers directly, so the call is one
    // launch and one sync instead of a copy in, the kernels, and up to four copies out.
    if (!sc16 && h->oneshot && h->zero_copy && h->one_ops && nd > 0 && rx_fb * (size_t)n_frames <= kZeroCopyBytes &&
        h->one_ops->split(n_frames, c.n_sym - 1, c.n_ant, h->n_sms, h->smem_optin) > 0) {
        void* a_rx = mapped_alias(h_rx);
        void* a_cb = mapped_alias(h_combined);
        void* a_bt = h_bits ? mapped_alias(h_bits) : nullptr;
        void* a_hc = h_hconj ? mapped_alias(h_hconj) : nullptr;
        void* a_hs = h_hsqrd ? mapped_alias(h_hsqrd) : nullptr;
        const bool aligned = ((reinterpret_cast<uintptr_t>(a_rx) | reinterpret_cast<uintptr_t>(a_cb) | reinterpret_cast<uintptr_t>(a_hc)) %
                              sizeof(float2)) == 0 && reinterpret_cast<uintptr_t>(a_hs) % sizeof(float) == 0;
        if (aligned && a_rx && a_cb && (!h_bits || a_bt) && (!h_hconj || a_hc) && (!h_hsqrd || a_hs)) {
            cudaStream_t st = compute_stream(h);
            int rc0 = ensure_chan(h, h->dev_ch, n_frames, st);
            if (rc0 != LSMRC_OK) return rc0;
            rc0 = launch_frames(h, st, static_cast<const float2*>(a_rx), n_frames, h->dev_ch, static_cast<float2*>(a_hc),
                                static_cast<float*>(a_hs), static_cast<float2*>(a_cb), static_cast<uint8_t*>(a_bt), false);
            if (rc0 != LSMRC_OK) return rc0;
            CK(h, cudaStreamSynchronize(st));
            h->zero_copy_calls++;
            return LSMRC_OK;
        }
    }
    int rc = ensure_lanes(h);
    if (rc != LSMRC_OK) return rc;
    const size_t hc_fb = (size_t)c.n_ant * h->K * sizeof(float2);
    const size_t hs_fb = (size_t)h->K * sizeof(float);
    const size_t cb_fb = nd * h->K * sizeof(float2);
    const size_t bt_fb = nd * h->row_bytes;
    ScopedPin pin_rx, pin_hc, pin_hs, pin_cb, pin_bt;
    pin_rx.pin(h_rx, rx_fb * n_frames);
    pin_hc.pin(h_hconj, hc_fb * n_frames);
    pin_hs.pin(h_hsqrd, hs_fb * n_frames);
    pin_cb.pin(h_combined, cb_fb * n_frames);
    pin_bt.pin(h_bits, bt_fb * n_frames);

    // strided H2D that skips the cyclic prefix: worth it when rows are long enough for the copy engine
    const bool strip_cp = sc16 ? (h->h2d_strip_cp && c.cp_len > 0 && (size_t)c.fft_size * elem >= h->h2d_strip_min_row) : strip_cp_on_h2d(h);
    if (sc16)
        for (Lane& L : h->lanes)
            if (!L.d_rx16) CK(h, cudaMalloc(&L.d_rx16, (size_t)c.max_frames * h->frame_elems * sizeof(short2)));
    int chunk_idx = 0;
    for (int f0 = 0; f0 < n_frames; f0 += c.max_frames, ++chunk_idx) {
        const int nf = (n_frames - f0 < c.max_frames) ? (n_frames - f0) : c.max_frames;
        Lane& L = h->lanes[(size_t)chunk_idx % h->lanes.size()];
        const char* src = static_cast<const char*>(h_rx) + (size_t)f0 * rx_fb;
        RxLayout dense_lay{};
        dense_lay.dense = true;
        void* d_in = sc16 ? static_cast<void*>(L.d_rx16) : static_cast<void*>(L.d_rx);
        const long long n_rows = (long long)nf * c.n_sym * c.n_ant;
        if (strip_cp) {
            // the cyclic prefix is never used: leave it on the host (C/(N+C) of the PCIe bytes)
            const size_t row = (size_t)c.fft_size * elem, pitch = (size_t)(c.fft_size + c.cp_len) * elem;
            CK(h, cudaMemcpy2DAsync(d_in, row, src + (size_t)c.cp_len * elem, pitch, row, (size_t)n_rows, cudaMemcpyHostToDevice, L.st));
        } else {
            CK(h, cudaMemcpyAsync(d_in, src, rx_fb * nf, cudaMemcpyHostToDevice, L.st));
        }
        if (sc16) {
            // wire format -> complex float on the device, always into dense rows (what is left of the prefix goes here)
            rc = launch_sc16_to_fc32(h, L.st, L.d_rx, L.d_rx16, n_rows, strip_cp ? c.fft_size : c.fft_size + c.cp_len,
                                     strip_cp ? 0 : c.cp_len, c.fft_size, scale);
            if (rc != LSMRC_OK) return rc;
        }
        rc = launch_frames(h, L.st, L.d_rx, nf, L.ch, h_hconj ? L.d_hconj : nullptr, nullptr, L.d_comb,
                           h_bits ? L.d_bits : nullptr, false, (strip_cp || sc16) ? &dense_lay : nullptr);
        if (rc != LSMRC_OK) return rc;
        if (nd > 0)
            CK(h, cudaMemcpyAsync(static_cast<char*>(h_combined) + (size_t)f0 * cb_fb, L.d_comb, cb_fb * nf,
                                  cudaMemcpyDeviceToHost, L.st));
        if (h_bits && nd > 0)
            CK(h, cudaMemcpyAsync(static_cast<char*>(h_bits) + (size_t)f0 * bt_fb, L.d_bits, bt_fb * nf,
                                  cudaMemcpyDeviceToHost, L.st));
        if (h_hconj)
            CK(h, cudaMemcpyAsync(static_cast<char*>(h_hconj) + (size_t)f0 * hc_fb, L.d_hconj, hc_fb * nf,
                                  cudaMemcpyDeviceToHost, L.st));
        if (h_hsqrd)
            CK(h, cudaMemcpyAsync(static_cast<char*>(h_hsqrd) + (size_t)f0 * hs_fb, L.ch.hsqrd, hs_fb * nf,
                                  cudaMemcpyDeviceToHost, L.st));
    }
    for (Lane& L : h->lanes) CK(h, cudaStreamSynchronize(L.st));
    return LSMRC_OK;
}

int lsmrc_demod_frames_host(lsmrc_handle h, const void* h_rx, int n_frames, void* h_hconj, void* h_hsqrd,
                            void* h_combined, void* h_bits)
{
    return demod_frames_host_impl(h, h_rx, n_frames, h_hconj, h_hsqrd, h_combined, h_bits, false, 1.f);
}

int lsmrc_demod_frames_host_sc16(lsmrc_handle h, const int16_t* h_rx_iq, int n_frames, float scale, void* h_hconj, void* h_hsqrd,
                                 void* h_combined, void* h_bits)
{
    return demod_frames_host_impl(h, h_rx_iq, n_frames, h_hconj, h_hsqrd, h_combined, h_bits, true, scale);
}

int lsmrc_sc16_to_fc32_device(lsmrc_handle h, const int16_t* d_iq, long long rows, int row_len_in, int skip, int row_len_out, float scale,
                              void* d_out)
{
    if (!h || !d_iq || !d_out) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (rows < 0 || row_len_out < 0 || skip < 0 || (long long)skip + row_len_out > row_len_in) return fail(h, LSMRC_ERR_INVALID, "bad row geometry");
    if (rows == 0 || row_len_out == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    return launch_sc16_to_fc32(h, compute_stream(h), static_cast<float2*>(d_out), reinterpret_cast<const short2*>(d_iq), rows, row_len_in, skip,
                               row_len_out, scale);
}

int lsmrc_first_vector(lsmrc_handle h, const void* rx_sym, int on_device)
{
    if (!h || !rx_sym) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    CK(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_symbol_state(h);
    if (rc != LSMRC_OK) return rc;
    const float2* d_in = nullptr;
    if ((rc = stage_symbol(h, rx_sym, on_device, &d_in)) != LSMRC_OK) return rc;
    KernelParams p = base_params(h);
    p.rx = d_in;
    p.frame_stride = 0;
    p.sym_stride = 0;
    p.n_frames = 1;
    if ((rc = launch_pilot(h, h->own_stream, p, h->one_ch, h->d_one_hconj, nullptr)) != LSMRC_OK) return rc;
    h->have_channel = true;
    return LSMRC_OK;
}

int lsmrc_demod_one_symbol(lsmrc_handle h, const void* rx_sym, int on_device, void* h_combined, void* h_bits)
{
    if (!h || !rx_sym || !h_combined) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (!h->have_channel) return fail(h, LSMRC_ERR_STATE, "lsmrc_first_vector must run before lsmrc_demod_one_symbol");
    CK(h, cudaSetDevice(h->cfg.device));
    const float2* d_in = nullptr;
    int rc = stage_symbol(h, rx_sym, on_device, &d_in);
    if (rc != LSMRC_OK) return rc;
    KernelParams p = base_params(h);
    p.rx = d_in;
    p.frame_stride = 0;
    p.sym_stride = 0;
    p.n_frames = 1;
    p.combined = h->d_one_comb;
    p.bits = h->d_one_bits;
    cudaStream_t st = h->own_stream;
    if ((rc = launch_data(h, st, p, h->one_ch, nullptr, 0, 1)) != LSMRC_OK) return rc;
    CK(h, cudaMemcpyAsync(h->h_one_comb, h->d_one_comb, (size_t)h->K * sizeof(float2), cudaMemcpyDeviceToHost, st));
    if (h_bits) CK(h, cudaMemcpyAsync(h->h_one_bits, h->d_one_bits, h->row_bytes, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    std::memcpy(h_combined, h->h_one_comb, (size_t)h->K * sizeof(float2));
    if (h_bits) std::memcpy(h_bits, h->h_one_bits, h->row_bytes);
    return LSMRC_OK;
}

int lsmrc_get_channel(lsmrc_handle h, void* h_hconj, void* h_hsqrd)
{
    if (!h) return LSMRC_ERR_INVALID;
    if (!h->have_channel) return fail(h, LSMRC_ERR_STATE, "no channel estimate yet");
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->own_stream));
    if (h_hconj) CK(h, cudaMemcpy(h_hconj, h->d_one_hconj, (size_t)h->cfg.n_ant * h->K * sizeof(float2), cudaMemcpyDeviceToHost));
    if (h_hsqrd) CK(h, cudaMemcpy(h_hsqrd, h->one_ch.hsqrd, (size_t)h->K * sizeof(float), cudaMemcpyDeviceToHost));
    return LSMRC_OK;
}

int lsmrc_get_channel_device(lsmrc_handle h, void* d_hconj, void* d_hsqrd)
{
    if (!h) return LSMRC_ERR_INVALID;
    if (!h->have_channel) return fail(h, LSMRC_ERR_STATE, "no channel estimate yet");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = h->own_stream;
    if (d_hconj)
        CK(h, cudaMemcpyAsync(d_hconj, h->d_one_hconj, (size_t)h->cfg.n_ant * h->K * sizeof(float2), cudaMemcpyDeviceToDevice, st));
    if (d_hsqrd)
        CK(h, cudaMemcpyAsync(d_hsqrd, h->one_ch.hsqrd, (size_t)h->K * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CK(h, cudaStreamSynchronize(st));
    return LSMRC_OK;
}

// ---- ring lanes -----------------------------------------------------------------------

// first event of a submission's timeline; the very first submission of the handle also defines time zero
static cudaError_t ring_mark_start(lsmrc_ctx* h, Lane& L)
{
    if (!h->ring_epoch) {
        cudaError_t e = cudaEventCreate(&h->ring_epoch);
        if (e != cudaSuccess) return e;
        if ((e = cudaEventRecord(h->ring_epoch, L.st)) != cudaSuccess) return e;
    }
    return cudaEventRecord(L.t_start, L.st);
}

// H2D of n_slots consecutive ring slots into the lane's staging tensor starting at slot position `at`: the slots are one
// uniform [n_slots * A][N + C] array, so leaving the prefix behind is a single strided copy.
static int ring_copy_slots(lsmrc_ctx* h, Lane& L, const void* h_slots, int at, int n_slots, bool strip)
{
    const lsmrc_config& c = h->cfg;
    if (n_slots <= 0) return LSMRC_OK;
    if (strip) {
        const size_t row = (size_t)c.fft_size * sizeof(float2), pitch = (size_t)(c.fft_size + c.cp_len) * sizeof(float2);
        CK(h, cudaMemcpy2DAsync(reinterpret_cast<char*>(L.d_rx) + (size_t)at * c.n_ant * row, row,
                                static_cast<const char*>(h_slots) + (size_t)c.cp_len * sizeof(float2), pitch, row, (size_t)n_slots * c.n_ant,
                                cudaMemcpyHostToDevice, L.st));
    } else {
        const size_t slot_bytes = h->slot_elems * sizeof(float2);
        CK(h, cudaMemcpyAsync(reinterpret_cast<char*>(L.d_rx) + (size_t)at * slot_bytes, h_slots, slot_bytes * n_slots, cudaMemcpyHostToDevice, L.st));
    }
    return LSMRC_OK;
}

static int ring_enqueue_compute(lsmrc_ctx* h, Lane& L, int n_frames, bool dense = false)
{
    const lsmrc_config& c = h->cfg;
    const size_t nd = (size_t)(c.n_sym - 1);
    CK(h, cudaEventRecord(L.copied, L.st));
    RxLayout dense_lay{};
    dense_lay.dense = true;
    int rc = launch_frames(h, L.st, L.d_rx, n_frames, L.ch, L.d_hconj, nullptr, L.d_comb, L.d_bits, false, dense ? &dense_lay : nullptr);
    if (rc != LSMRC_OK) return rc;
    CK(h, cudaEventRecord(L.t_kernels, L.st));
    if (nd > 0) {
        CK(h, cudaMemcpyAsync(L.h_comb, L.d_comb, n_frames * nd * h->K * sizeof(float2), cudaMemcpyDeviceToHost, L.st));
        CK(h, cudaMemcpyAsync(L.h_bits, L.d_bits, n_frames * nd * h->row_bytes, cudaMemcpyDeviceToHost, L.st));
    }
    CK(h, cudaMemcpyAsync(L.h_hconj, L.d_hconj, n_frames * (size_t)c.n_ant * h->K * sizeof(float2), cudaMemcpyDeviceToHost, L.st));
    CK(h, cudaEventRecord(L.done, L.st));
    L.busy = true;
    L.ring_frames = n_frames;
    return LSMRC_OK;
}

// Small frame in a pinned ring: the one-launch kernel reads the slots where they lie and writes the lane's pinned
// result buffers directly -- no copy in, no copies out.  Returns 1 when it took the frame, 0 when the staged
// path has to (pageable ring, large frame, one-launch kernel not applicable), < 0 on error.
static int ring_try_in_place(lsmrc_ctx* h, Lane& L, const void* h_first, int n_first, const void* h_second, size_t slot_stride_bytes,
                             int n_frames = 1)
{
    const lsmrc_config& c = h->cfg;
    if (!(h->oneshot && h->zero_copy && h->one_ops) || c.n_sym < 2 || h->frame_elems * sizeof(float2) * n_frames > kZeroCopyBytes) return 0;
    const int n_slots = n_frames * c.n_sym;
    if (slot_stride_bytes % sizeof(float2) != 0) return 0;
    if ((reinterpret_cast<uintptr_t>(h_first) | reinterpret_cast<uintptr_t>(h_second)) % sizeof(float) != 0) return 0;
    if (h->one_ops->split(n_frames, c.n_sym - 1, c.n_ant, h->n_sms, h->smem_optin) <= 0) return 0;
    void* a1 = mapped_alias(h_first);
    void* a2 = (n_first < n_slots) ? mapped_alias(h_second) : nullptr;
    if (!a1 || (n_first < n_slots && !a2)) return 0;
    if (!L.a_comb) {
        L.a_comb = static_cast<float2*>(mapped_alias(L.h_comb));
        L.a_bits = static_cast<uint8_t*>(mapped_alias(L.h_bits));
        L.a_hconj = static_cast<float2*>(mapped_alias(L.h_hconj));
    }
    if (!L.a_comb || !L.a_bits || !L.a_hconj) return 0;
    RxLayout lay;
    lay.dense = false;
    lay.sym_stride = (long long)(slot_stride_bytes / sizeof(float2));
    lay.rx2 = a2 ? static_cast<const float2*>(a2) : static_cast<const float2*>(a1);  // (unused when the run does not wrap)
    lay.split_sym = n_first < n_slots ? n_first : n_slots;
    lay.align4 = ((reinterpret_cast<uintptr_t>(a1) | reinterpret_cast<uintptr_t>(a2)) % sizeof(float2)) != 0;
    const int rc = launch_frames(h, L.st, static_cast<const float2*>(a1), n_frames, L.ch, L.a_hconj, nullptr, L.a_comb, L.a_bits, false, &lay);
    if (rc != LSMRC_OK) return rc;
    CK(h, cudaEventRecord(L.copied, L.st));  // the slots are free once the kernel has read them
    CK(h, cudaEventRecord(L.t_kernels, L.st));
    CK(h, cudaEventRecord(L.done, L.st));
    L.busy = true;
    L.ring_frames = n_frames;
    h->zero_copy_calls++;
    return 1;
}

int lsmrc_ring_prepare(lsmrc_handle h)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    return ensure_lanes(h);
}

int lsmrc_ring_submit_frame(lsmrc_handle h, int lane, const void* h_slots, size_t slot_stride_bytes)
{
    if (!h || !h_slots) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    if (lane < 0 || lane >= h->cfg.n_lanes) return fail(h, LSMRC_ERR_INVALID, "lane out of range");
    CK(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lanes(h);
    if (rc != LSMRC_OK) return rc;
    Lane& L = h->lanes[(size_t)lane];
    const size_t slot_bytes = h->slot_elems * sizeof(float2);
    if (slot_stride_bytes < slot_bytes) return fail(h, LSMRC_ERR_INVALID, "slot stride smaller than a slot");
    CK(h, ring_mark_start(h, L));
    if ((rc = ring_try_in_place(h, L, h_slots, h->cfg.n_sym, nullptr, slot_stride_bytes)) != 0) return rc < 0 ? rc : LSMRC_OK;
    if (slot_stride_bytes == slot_bytes) {
        const bool strip = strip_cp_on_h2d(h);
        if ((rc = ring_copy_slots(h, L, h_slots, 0, h->cfg.n_sym, strip)) != LSMRC_OK) return rc;
        return ring_enqueue_compute(h, L, 1, strip);
    } else {
        CK(h, cudaMemcpy2DAsync(L.d_rx, slot_bytes, h_slots, slot_stride_bytes, slot_bytes, (size_t)h->cfg.n_sym,
                                cudaMemcpyHostToDevice, L.st));
    }
    return ring_enqueue_compute(h, L, 1);
}

int lsmrc_ring_submit_frames(lsmrc_handle h, int lane, const void* h_first, int n_first, const void* h_second, int n_frames)
{
    if (!h || !h_first) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (!h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first");
    if (lane < 0 || lane >= h->cfg.n_lanes) return fail(h, LSMRC_ERR_INVALID, "lane out of range");
    if (n_frames < 1 || n_frames > h->cfg.max_frames) return fail(h, LSMRC_ERR_INVALID, "n_frames must be in 1..max_frames");
    const int n_slots = n_frames * h->cfg.n_sym;
    if (n_first < 0 || n_first > n_slots || (n_first < n_slots && !h_second)) return fail(h, LSMRC_ERR_INVALID, "bad split");
    CK(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lanes(h);
    if (rc != LSMRC_OK) return rc;
    Lane& L = h->lanes[(size_t)lane];
    const size_t slot_bytes = h->slot_elems * sizeof(float2);
    CK(h, ring_mark_start(h, L));
    if (n_first > 0 && (rc = ring_try_in_place(h, L, h_first, n_first, h_second, slot_bytes, n_frames)) != 0) return rc < 0 ? rc : LSMRC_OK;
    const bool strip = strip_cp_on_h2d(h);  // the cyclic prefix is never used: leave it in the ring (C/(N+C) of the PCIe bytes)
    if ((rc = ring_copy_slots(h, L, h_first, 0, n_first, strip)) != LSMRC_OK) return rc;
    if ((rc = ring_copy_slots(h, L, h_second, n_first, n_slots - n_first, strip)) != LSMRC_OK) return rc;
    return ring_enqueue_compute(h, L, n_frames, strip);
}

int lsmrc_ring_submit_split(lsmrc_handle h, int lane, const void* h_first, int n_first, const void* h_second)
{
    return lsmrc_ring_submit_frames(h, lane, h_first, n_first, h_second, 1);
}

int lsmrc_ring_copy_done(lsmrc_handle h, int lane)
{
    if (!h || lane < 0 || lane >= (int)h->lanes.size()) return fail(h, LSMRC_ERR_INVALID, "lane out of range");
    CK(h, cudaEventSynchronize(h->lanes[(size_t)lane].copied));
    return LSMRC_OK;
}

int lsmrc_ring_copy_query(lsmrc_handle h, int lane)
{
    if (!h || lane < 0 || lane >= (int)h->lanes.size()) return fail(h, LSMRC_ERR_INVALID, "lane out of range");
    const cudaError_t e = cudaEventQuery(h->lanes[(size_t)lane].copied);
    if (e == cudaSuccess) return 1;
    if (e == cudaErrorNotReady) {
        cudaGetLastError();
        return 0;
    }
    return fail_cuda(h, e, "cudaEventQuery");
}

int lsmrc_ring_wait(lsmrc_handle h, int lane, const void** combined, const void** bits, const void** hconj)
{
    if (!h || lane < 0 || lane >= (int)h->lanes.size()) return fail(h, LSMRC_ERR_INVALID, "lane out of range");
    Lane& L = h->lanes[(size_t)lane];
    if (!L.busy) return fail(h, LSMRC_ERR_STATE, "lane has nothing in flight");
    CK(h, cudaEventSynchronize(L.done));
    L.busy = false;
    if (combined) *combined = L.h_comb;
    if (bits) *bits = L.h_bits;
    if (hconj) *hconj = L.h_hconj;
    return LSMRC_OK;
}

int lsmrc_ring_trace(lsmrc_handle h, int lane, float* ms4)
{
    if (!h || !ms4 || lane < 0 || lane >= (int)h->lanes.size()) return fail(h, LSMRC_ERR_INVALID, "bad argument");
    Lane& L = h->lanes[(size_t)lane];
    if (!h->ring_epoch || L.busy) return fail(h, LSMRC_ERR_STATE, "collect the lane with lsmrc_ring_wait first");
    cudaEvent_t ev[4] = {L.t_start, L.copied, L.t_kernels, L.done};
    for (int i = 0; i < 4; ++i) CK(h, cudaEventElapsedTime(&ms4[i], h->ring_epoch, ev[i]));
    return LSMRC_OK;
}

// ---- stand-alone steps (the kernel-wrapper methods of gpuLS.cuh:87-99) -------------------------------

static unsigned ew_grid(long long n) { long long g = (n + 255) / 256; return (unsigned)(g < 1 ? 1 : (g > 148 * 16 ? 148 * 16 : g)); }

int lsmrc_stage_drop_prefix(lsmrc_handle h, void* d_out, const void* d_in, long long rows)
{
    if (!h || !d_out || !d_in || rows < 0) return fail(h, LSMRC_ERR_INVALID, "bad argument");
    if (rows == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    k_drop_prefix<<<ew_grid(rows * h->cfg.fft_size), 256, 0, compute_stream(h)>>>(
        static_cast<float2*>(d_out), static_cast<const float2*>(d_in), rows, h->cfg.fft_size, h->cfg.cp_len);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_stage_fft(lsmrc_handle h, void* d_rows, long long rows)
{
    if (!h || !d_rows || rows < 0 || rows > 0x7fffffffLL) return fail(h, LSMRC_ERR_INVALID, "bad argument");
    if (rows == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    KernelParams p = base_params(h);
    p.rx = static_cast<const float2*>(d_rows);
    p.combined = static_cast<float2*>(d_rows);
    p.ant_stride = h->cfg.fft_size;
    p.cp = 0;
    p.n_frames = (int)rows;
    CK(h, h->ops->launch(MODE_FFT, p, compute_stream(h), h->max_data_ctas));
    h->launches++;
    return LSMRC_OK;
}

int lsmrc_stage_find_hs(lsmrc_handle h, const void* d_yfft, void* d_hconj, const void* d_x)
{
    if (!h || !d_yfft || !d_hconj) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (!d_x && !h->have_pilot) return fail(h, LSMRC_ERR_NO_PILOT, "set the pilot first or pass dX");
    CK(h, cudaSetDevice(h->cfg.device));
    const int A = h->cfg.n_ant, N = h->cfg.fft_size;
    k_find_hs<<<ew_grid((long long)A * h->K), 256, 0, compute_stream(h)>>>(
        static_cast<const float2*>(d_yfft), static_cast<float2*>(d_hconj),
        d_x ? static_cast<const float2*>(d_x) : h->d_pilot_bin, A, N, d_x ? h->K : 0);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_stage_find_hsqrd(lsmrc_handle h, const void* d_hconj, void* d_hsqrd)
{
    if (!h || !d_hconj || !d_hsqrd) return fail(h, LSMRC_ERR_INVALID, "null argument");
    CK(h, cudaSetDevice(h->cfg.device));
    k_find_hsqrd<<<ew_grid(h->K), 256, 0, compute_stream(h)>>>(static_cast<const float2*>(d_hconj),
                                                               static_cast<float*>(d_hsqrd), h->cfg.n_ant, h->K);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_stage_mult_conj(lsmrc_handle h, const void* d_yfft, const void* d_hconj, void* d_yf, int n_syms)
{
    if (!h || !d_yfft || !d_hconj || !d_yf || n_syms < 0) return fail(h, LSMRC_ERR_INVALID, "bad argument");
    if (n_syms == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    k_mult_conj<<<ew_grid((long long)n_syms * h->cfg.n_ant * h->K), 256, 0, compute_stream(h)>>>(
        static_cast<const float2*>(d_yfft), static_cast<const float2*>(d_hconj), static_cast<float2*>(d_yf), n_syms,
        h->cfg.n_ant, h->cfg.fft_size);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_stage_combine(lsmrc_handle h, const void* d_yf, const void* d_hsqrd, void* d_out, int n_syms)
{
    if (!h || !d_yf || !d_hsqrd || !d_out || n_syms < 0) return fail(h, LSMRC_ERR_INVALID, "bad argument");
    if (d_out == d_yf) return fail(h, LSMRC_ERR_INVALID, "d_out must not alias d_yf (the reference's in-place form races, gpuLS.cu:244-256)");
    if (n_syms == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    k_combine<<<ew_grid((long long)n_syms * h->K), 256, 0, compute_stream(h)>>>(
        static_cast<const float2*>(d_yf), static_cast<const float*>(d_hsqrd), static_cast<float2*>(d_out), n_syms,
        h->cfg.n_ant, h->K);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_stage_shift_rows(lsmrc_handle h, const void* d_in, void* d_out, long long rows)
{
    if (!h || !d_in || !d_out || rows < 0) return fail(h, LSMRC_ERR_INVALID, "bad argument");
    if (d_in == d_out) return fail(h, LSMRC_ERR_INVALID, "d_out must not alias d_in");
    if (rows == 0) return LSMRC_OK;
    CK(h, cudaSetDevice(h->cfg.device));
    k_shift_rows<<<ew_grid(rows * h->K), 256, 0, compute_stream(h)>>>(static_cast<const float2*>(d_in),
                                                                       static_cast<float2*>(d_out), rows, h->K);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

// ---- receive front end before the hot path (rx_and_corr.cpp:332-393) ---------------------------------------

int lsmrc_sync_correlate(lsmrc_handle h, const void* d_buf, int n_chan, int samps, const void* d_pn, int pn_len,
                         float thres, int* offset, int* chan, float* metric, void* d_metric_all)
{
    if (!h || !d_buf || !d_pn || !offset) return fail(h, LSMRC_ERR_INVALID, "null argument");
    if (n_chan < 1 || pn_len < 1 || samps < pn_len || pn_len > 4096) return fail(h, LSMRC_ERR_INVALID, "bad sizes");
    if ((long long)n_chan * samps >= (1LL << 31)) return fail(h, LSMRC_ERR_INVALID, "capture too long");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = compute_stream(h);
    if (!h->d_hit) CK(h, cudaMalloc(&h->d_hit, sizeof(unsigned long long)));
    CK(h, cudaMemsetAsync(h->d_hit, 0xff, sizeof(unsigned long long), st));
    const int n_off = samps - pn_len + 1;
    dim3 grid((unsigned)((n_off + kSyncThreads - 1) / kSyncThreads), (unsigned)n_chan);
    const size_t smem = sizeof(float2) * (size_t)(pn_len + kSyncThreads + pn_len - 1);
    k_sync_correlate<<<grid, kSyncThreads, smem, st>>>(static_cast<const float2*>(d_buf), samps,
                                                      static_cast<const float2*>(d_pn), pn_len, thres, h->d_hit,
                                                      static_cast<float*>(d_metric_all));
    h->launches++;
    CK(h, cudaGetLastError());
    unsigned long long key = 0;
    CK(h, cudaMemcpyAsync(&key, h->d_hit, sizeof(key), cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    if (key == ~0ULL) {
        *offset = -1;
        if (chan) *chan = -1;
        if (metric) *metric = 0.f;
        return LSMRC_OK;
    }
    const long long pos = (long long)(key >> 32);
    *offset = (int)(pos % samps);
    if (chan) *chan = (int)(pos / samps);
    if (metric) {
        const unsigned bits = (unsigned)(key & 0xffffffffu);
        std::memcpy(metric, &bits, sizeof(float));
    }
    return LSMRC_OK;
}

int lsmrc_sync_assemble(lsmrc_handle h, const void* d_buf1, const void* d_buf2, int samps, int offset, int pn_len,
                        void* d_rx_frame)
{
    if (!h || !d_buf1 || !d_buf2 || !d_rx_frame) return fail(h, LSMRC_ERR_INVALID, "null argument");
    const lsmrc_config& c = h->cfg;
    const long long frame = (long long)c.n_sym * (c.fft_size + c.cp_len);
    if (offset < 0 || pn_len < 0 || offset + pn_len > samps || (long long)samps - pn_len < frame)
        return fail(h, LSMRC_ERR_INVALID, "capture buffer shorter than PN + one frame, or bad offset");
    CK(h, cudaSetDevice(h->cfg.device));
    k_sync_assemble<<<ew_grid(frame * c.n_ant), 256, 0, compute_stream(h)>>>(
        static_cast<const float2*>(d_buf1), static_cast<const float2*>(d_buf2), samps, offset, pn_len,
        static_cast<float2*>(d_rx_frame), c.n_sym, c.n_ant, c.fft_size + c.cp_len);
    h->launches++;
    CK(h, cudaGetLastError());
    return LSMRC_OK;
}

int lsmrc_copy_device(lsmrc_handle h, void* d_dst, const void* d_src, size_t bytes)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, compute_stream(h)));
    return LSMRC_OK;
}

// ---- plumbing ---------------------------------------------------------------------------

int lsmrc_dev_alloc(lsmrc_handle h, size_t bytes, void** d_ptr)
{
    if (!h || !d_ptr) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMalloc(d_ptr, bytes));
    return LSMRC_OK;
}
int lsmrc_dev_free(lsmrc_handle h, void* d_ptr)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaFree(d_ptr));
    return LSMRC_OK;
}
int lsmrc_copy_to_device(lsmrc_handle h, void* d_dst, const void* h_src, size_t bytes)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice));
    return LSMRC_OK;
}
int lsmrc_copy_to_host(lsmrc_handle h, void* h_dst, const void* d_src, size_t bytes)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(compute_stream(h)));
    CK(h, cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return LSMRC_OK;
}
int lsmrc_host_alloc(lsmrc_handle h, size_t bytes, void** h_ptr)
{
    if (!h || !h_ptr) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMallocHost(h_ptr, bytes));
    return LSMRC_OK;
}
int lsmrc_host_free(lsmrc_handle h, void* h_ptr)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaFreeHost(h_ptr));
    return LSMRC_OK;
}
int lsmrc_host_register(lsmrc_handle h, void* h_ptr, size_t bytes)
{
    if (!h || !h_ptr) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaHostRegister(h_ptr, bytes, cudaHostRegisterDefault));
    return LSMRC_OK;
}
int lsmrc_host_unregister(lsmrc_handle h, void* h_ptr)
{
    if (!h || !h_ptr) return LSMRC_ERR_INVALID;
    CK(h, cudaHostUnregister(h_ptr));
    return LSMRC_OK;
}
int lsmrc_set_stream(lsmrc_handle h, void* cuda_stream)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    // the channel state of the device-resident path is shared by consecutive calls: drain the stream it was used on
    CK(h, cudaStreamSynchronize(compute_stream(h)));
    h->user_stream = static_cast<cudaStream_t>(cuda_stream);
    h->use_user_stream = cuda_stream != nullptr;  // NULL = back to the handle's own stream
    return LSMRC_OK;
}
int lsmrc_sync(lsmrc_handle h)
{
    if (!h) return LSMRC_ERR_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(compute_stream(h)));
    CK(h, cudaStreamSynchronize(h->own_stream));
    for (Lane& L : h->lanes) CK(h, cudaStreamSynchronize(L.st));
    return LSMRC_OK;
}
int lsmrc_set_oneshot(lsmrc_handle h, int enabled)
{
    if (!h) return LSMRC_ERR_INVALID;
    h->oneshot = enabled != 0;
    h->zero_copy = enabled != 1;  // 1 = fused kernel but staged copies; any other non-zero value = both
    return LSMRC_OK;
}

long long lsmrc_oneshot_count(lsmrc_handle h) { return h ? h->oneshot_calls : -1; }

int lsmrc_set_one_launch_frames(lsmrc_handle h, int enabled)
{
    if (!h) return LSMRC_ERR_INVALID;
    h->one_launch_frames = enabled != 0;
    return LSMRC_OK;
}

long long lsmrc_one_launch_frames_count(lsmrc_handle h) { return h ? h->fused_calls : -1; }

int lsmrc_set_mu_pilots(lsmrc_handle h, int layout)
{
    if (!h) return LSMRC_ERR_INVALID;
    if (layout != LSMRC_MU_PILOTS_TIME && layout != LSMRC_MU_PILOTS_COMB) return fail(h, LSMRC_ERR_INVALID, "unknown pilot layout");
    h->mu_pilots = layout;
    return LSMRC_OK;
}

int lsmrc_set_timing(lsmrc_handle h, int enabled)
{
    if (!h) return LSMRC_ERR_INVALID;
    h->timing = enabled != 0;
    return LSMRC_OK;
}
int lsmrc_kernel_ms_history(lsmrc_handle h, int max_n, float* pilot_ms, float* data_ms, int* n_out)
{
    if (!h || max_n < 0 || !n_out) return LSMRC_ERR_INVALID;
    long long n = h->ev_calls < lsmrc_ctx::kEvRing ? h->ev_calls : lsmrc_ctx::kEvRing;
    if (n > max_n) n = max_n;
    for (long long i = 0; i < n; ++i) {
        cudaEvent_t* ev = h->ev[(h->ev_calls - n + i) % lsmrc_ctx::kEvRing];
        CK(h, cudaEventSynchronize(ev[2]));
        float a = 0.f, b = 0.f;
        CK(h, cudaEventElapsedTime(&a, ev[0], ev[1]));
        CK(h, cudaEventElapsedTime(&b, ev[1], ev[2]));
        if (pilot_ms) pilot_ms[i] = a;
        if (data_ms) data_ms[i] = b;
    }
    *n_out = (int)n;
    return LSMRC_OK;
}
int lsmrc_last_kernel_ms(lsmrc_handle h, float* pilot_ms, float* data_ms)
{
    if (!h) return LSMRC_ERR_INVALID;
    if (h->ev_calls == 0) return fail(h, LSMRC_ERR_STATE, "no timed call yet (lsmrc_set_timing)");
    int n = 0;
    return lsmrc_kernel_ms_history(h, 1, pilot_ms, data_ms, &n);
}
long long lsmrc_launch_count(lsmrc_handle h) { return h ? h->launches : 0; }
int lsmrc_describe_plan(lsmrc_handle h, char* buf, size_t buf_len)
{
    if (!h || !buf || buf_len == 0) return LSMRC_ERR_INVALID;
    const PlanOps* o = h->ops;
    const OneshotOps* q = h->one_ops;
    std::snprintf(buf, buf_len, "N=%d P=%d R2=%d R3=%d teams=%d threads=%d smem=%zu minblocks=%d; one-launch P=%d R2=%d R3=%d teams=%d calls=%lld in-place-host=%lld; h2d=%s",
                  o->N, o->P, o->R2, o->R3, o->teams, o->threads, o->smem, o->minb, q ? q->P : 0, q ? q->R2 : 0, q ? q->R3 : 0,
                  q ? q->teams : 0, h->oneshot_calls, h->zero_copy_calls,
                  (h->h2d_strip_cp && h->cfg.cp_len > 0 && (size_t)h->cfg.fft_size * sizeof(float2) >= h->h2d_strip_min_row) ? "strip-cp" : "whole-slots");
    return LSMRC_OK;
}

}  // extern "C"
