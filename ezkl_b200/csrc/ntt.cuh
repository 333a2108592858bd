// ntt.cuh — internal interface of the BN254 Fr number-theoretic-transform engine (ntt.cu).
#pragma once
#include <map>
#include <vector>
#include "common.cuh"
#include "field.cuh"

namespace b200 {

// Twiddle tables for one (log_n, omega) pair, device resident.
struct NttPlan {
    uint32_t log_n = 0;
    Fr omega;                 // Montgomery form
    int npass = 0;
    int logm[3] = {0, 0, 0};
    Fr* d_tw[3] = {nullptr, nullptr, nullptr};   // per pass: (omega^(N/M))^k, k < M/2
    uint4* d_staged[3] = {nullptr, nullptr, nullptr};   // per pass: per-stage twiddles, planar (v2 kernel)
    Fr* d_full = nullptr;     // omega^e, e < N (log_n <= 22): single-multiply inter-pass twiddles
    Fr* d_lo = nullptr;       // omega^e, e < 2^lo_bits
    Fr* d_hi = nullptr;       // omega^(e << lo_bits), e < N >> lo_bits
    uint32_t lo_bits = 0;
};

static constexpr int NTT_SCALE_GEOMETRIC = 4;
struct NttScale {             // optional per-element scaling fused into the first load / last store
    int mode = 0;             // 0 none, 1 one constant (c[0]), 3 cycle c[i % 3], NTT_SCALE_GEOMETRIC (pre only) c^i
    Fr c[3];
    // geometric pre-scale c^i = lo[i & (2^lo_bits - 1)] * hi[i >> lo_bits] from two device power tables (coset-part transforms);
    // internal: not accepted from the ABI's scale modes, not supported by the sharded transform
    const Fr* lo = nullptr;
    const Fr* hi = nullptr;
    uint32_t lo_bits = 0;
};

struct NttContext {
    std::vector<NttPlan*> plans;
    NttPlan* get(uint32_t log_n, const Fr& omega, cudaStream_t st);
    void release();
};

// `plan` = NttContext::get(log_n, omega) obtained by the caller under its own lock (plans are immutable once built).
// dst[p][j] = post(j) * sum_{i < n_in} pre(i) * src[p][i] * omega^(i j),  j < 2^log_n, for p < batch polynomials.
// src has n_in <= 2^log_n valid elements per polynomial (rest treated as zero), tmp and dst hold 2^log_n each;
// dst may alias src (when n_in == 2^log_n and strides match); tmp must not alias either.
int ntt_run(NttPlan* plan, const Fr* d_src, size_t src_stride, size_t n_in, Fr* d_tmp, size_t tmp_stride, Fr* d_dst, size_t dst_stride,
            uint32_t log_n, const Fr& omega, const NttScale& pre, const NttScale& post, int batch, cudaStream_t st);
int ntt_launches_per_run(uint32_t log_n);
// host-built tables of NTT_SCALE_GEOMETRIC for c^i, i < 2^log_n: lo (2^geo_lo_bits(log_n) entries) then hi (2^(log_n - geo_lo_bits) entries)
uint32_t geo_lo_bits(uint32_t log_n);
size_t geo_table_len(uint32_t log_n);
void geo_table_fill(const Fr& c, uint32_t log_n, Fr* out);
// one transform split across devices in contiguous natural-order slices, exchanges fused into the passes (ntt.cu)
int ntt_run_sharded(NttPlan* const* plans, int ndev, const int* dev_ids, const Fr* const* src, Fr* const* tmp, Fr* const* dst, uint32_t log_n, const Fr& omega,
                    const NttScale& pre, const NttScale& post, uint64_t n_in, cudaStream_t* st, cudaEvent_t* ev);

}  // namespace b200
