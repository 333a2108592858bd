// ntt.cu — BN254 Fr number-theoretic transform for sm_100a.
//
// Replaces halo2_proofs arithmetic.rs best_fft and the EvaluationDomain transforms built on it (lagrange_to_coeff,
// coeff_to_extended, extended_to_coeff; UPSTREAM poly/domain.rs — in-tree user /root/reference/src/circuit/modules/
// polycommit.rs:52, and every column transform of create_proof / keygen_pk, src/pfsys/mod.rs:396,456).
// Semantics are best_fft's: natural-order in, natural-order out, out[j] = sum_i a[i] * omega^(i*j); arithmetic is exact,
// so any factorisation gives the reference's bytes.
//
// Factorisation: N = M1 * M2 (* M3), M <= 1024, one kernel pass per factor.
//   k_ntt_pass2 (default): 256-thread CTAs hold 1024 elements; every thread runs TWO stages of the radix-2 DIF network on a
//     register-resident quad per round, the first round loads global -> registers and the last stores registers -> global
//     (bit reversal, the inter-pass twiddle omega^(j * i_rest) from a full or two-level table, and the post-scale fused), the
//     per-stage twiddle table is staged into shared memory with cp.async.bulk (TMA) + mbarrier.
//   k_ntt_pass (v1): one radix-2 stage per shared-memory round trip; kept for tiny passes and as B200_NTT_V=1.
// Coset pre-scaling (zeta^(i mod 3)), zero padding and the 1/N (and zeta^-(i mod 3)) post-scaling of the extended-domain
// transforms are fused into the first load / last store, and so is the geometric pre-scale c^i of a coset-part transform
// (coeff_to_extended_part: c = zeta * ext_omega^r, from two host-built power tables; a separate kernel instantiation).
// Algorithmic HBM traffic: 64 B per element per transform; this schedule moves 64 B per element per PASS (2 passes up to
// 2^20, 3 above).  The kernels are bound by the 254-bit multiply (10-15 per element), not by HBM: see DESIGN.md §4.3.
#include <cstdlib>
#include "ntt.cuh"

namespace b200 {

struct PassArgs {
    const Fr* src; Fr* dst;
    size_t src_pstride, dst_pstride;
    uint32_t logm, log_g, inner_cnt, in_r_fast;
    uint64_t in_rs, in_inner_s, in_outer_s;
    uint64_t out_rs, out_inner_s, out_outer_s;
    uint64_t n_in;
    uint32_t tw_on, rest_is_inner, lo_bits, first, last;
    uint64_t tw_mul;
    const Fr* tw_m; const Fr* t_lo; const Fr* t_hi;
    const uint4* tw_staged;      // v2: per-stage twiddles, planar [2][M] (lo plane, hi plane), stage s at offset 2^s - 1
    const Fr* t_full;            // v2: omega^e for every e < N (single-multiply inter-pass twiddle), or null
    NttScale pre, post;
    // sharded transform (one polynomial split across devices in contiguous natural-order slices of 2^log_slice elements):
    // element idx of the distributed source / destination lives at peers[idx >> log_slice][idx & (2^log_slice - 1)], reached by
    // ordinary loads / stores on peer-mapped pointers (NVLink), so the exchange steps of the six-step scheme are fused into the passes
    uint32_t peer_on, log_slice, block0;
    const Fr* src_peers[8];
    Fr* dst_peers[8];
};

DEV Fr sh_get(const uint4* lo, const uint4* hi, uint32_t i) {
    uint4 a = lo[i], b = hi[i];
    Fr r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w; r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
DEV void sh_put(uint4* lo, uint4* hi, uint32_t i, const Fr& v) {
    lo[i] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    hi[i] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

// c^idx of the geometric pre-scale: two table loads, one multiplication
DEV Fr geo_power(const NttScale& s, uint64_t idx) {
    return fp_load(s.lo + (idx & ((1ull << s.lo_bits) - 1))) * fp_load(s.hi + (idx >> s.lo_bits));
}

// GEO: the first load applies NTT_SCALE_GEOMETRIC; a separate instantiation, so the other modes keep their code unchanged
template <bool GEO>
__global__ void __launch_bounds__(1024, 1) k_ntt_pass(const PassArgs a) {
    extern __shared__ uint4 sh[];
    const uint32_t M = 1u << a.logm, G = 1u << a.log_g, total = M << a.log_g;
    uint4* dlo = sh; uint4* dhi = sh + total; uint4* tlo = sh + 2 * total; uint4* thi = tlo + (M >> 1);
    const uint32_t tid = threadIdx.x, nt = blockDim.x;
    const uint32_t tiles_per_outer = a.inner_cnt >> a.log_g;
    const uint32_t outer = blockIdx.x / tiles_per_outer, tile = blockIdx.x % tiles_per_outer;
    const uint32_t inner0 = tile << a.log_g;
    const Fr* src = a.src + (size_t)blockIdx.y * a.src_pstride;
    Fr* dst = a.dst + (size_t)blockIdx.y * a.dst_pstride;
    const uint64_t in_base = (uint64_t)outer * a.in_outer_s + (uint64_t)inner0 * a.in_inner_s;
    const uint64_t out_base = (uint64_t)outer * a.out_outer_s + (uint64_t)inner0 * a.out_inner_s;

    for (uint32_t k = tid; k < (M >> 1); k += nt) { Fr w = fp_load(a.tw_m + k); sh_put(tlo, thi, k, w); }
    for (uint32_t e = tid; e < total; e += nt) {
        uint32_t g, r;
        if (a.in_r_fast) { r = e & (M - 1); g = e >> a.logm; } else { g = e & (G - 1); r = e >> a.log_g; }
        const uint64_t idx = in_base + (uint64_t)g * a.in_inner_s + (uint64_t)r * a.in_rs;
        Fr v = fp_zero<FrTag>();
        if (idx < a.n_in) {
            v = fp_load(src + idx);
            if (a.first) {
                if constexpr (GEO) v = v * geo_power(a.pre, idx);
                else if (a.pre.mode == 1) v = v * a.pre.c[0];
                else if (a.pre.mode == 3) { uint32_t m3 = (uint32_t)(idx % 3); if (m3) v = v * a.pre.c[m3]; }
            }
        }
        sh_put(dlo, dhi, (g << a.logm) + r, v);
    }
    __syncthreads();
    // radix-2 decimation-in-frequency: natural order in, bit-reversed order out
    const uint32_t nbf = total >> 1;
    for (int s = (int)a.logm - 1; s >= 0; --s) {
        const uint32_t half = 1u << s;
        for (uint32_t bf = tid; bf < nbf; bf += nt) {
            const uint32_t g = bf >> (a.logm - 1), b = bf & ((M >> 1) - 1);
            const uint32_t j = b & (half - 1);
            const uint32_t i0 = (g << a.logm) + ((b >> s) << (s + 1)) + j, i1 = i0 + half;
            Fr x = sh_get(dlo, dhi, i0), y = sh_get(dlo, dhi, i1);
            Fr sum = x + y, dif = x - y;
            if (s > 0) { Fr w = sh_get(tlo, thi, j << (a.logm - 1 - s)); dif = dif * w; }
            sh_put(dlo, dhi, i0, sum);
            sh_put(dlo, dhi, i1, dif);
        }
        __syncthreads();
    }
    for (uint32_t e = tid; e < total; e += nt) {
        const uint32_t g = e & (G - 1), rp = e >> a.log_g;
        const uint32_t pos = a.logm ? (__brev(rp) >> (32 - a.logm)) : 0;
        Fr v = sh_get(dlo, dhi, (g << a.logm) + pos);
        if (a.tw_on) {
            const uint64_t i_rest = a.rest_is_inner ? (uint64_t)(inner0 + g) : 0;
            const uint64_t ex = a.tw_mul * (uint64_t)rp * i_rest;
            if (ex) {
                const uint32_t elo = (uint32_t)(ex & ((1ull << a.lo_bits) - 1)), ehi = (uint32_t)(ex >> a.lo_bits);
                Fr w = fp_load(a.t_lo + elo);
                if (ehi) w = w * fp_load(a.t_hi + ehi);
                v = v * w;
            }
        }
        const uint64_t idx = out_base + (uint64_t)g * a.out_inner_s + (uint64_t)rp * a.out_rs;
        if (a.last) {
            if (a.post.mode == 1) v = v * a.post.c[0];
            else if (a.post.mode == 3) v = v * a.post.c[(uint32_t)(idx % 3)];
        }
        fp_store(dst + idx, v);
    }
}


// ---- v2 pass: radix-4 butterflies in registers, one shared-memory exchange per TWO stages --------------------------------
// Each thread owns one "quad" {p, p+q, p+2q, p+3q} per round and runs stages s and s-1 of the DIF network on it in
// registers (an odd log M starts with a single-stage round on the same quad shape).  The first round loads straight from
// global memory into registers and the last round stores straight from registers to global memory (bit-reversal, inter-pass
// twiddle and post-scale fused), so an M-point line touches shared memory ceil(log M / 2) - 1 times instead of log M.
// The per-stage twiddle table is staged into shared memory by the TMA engine (cp.async.bulk + mbarrier, SASS UBLKCP) while
// the first round's global loads are in flight.
DEV uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
DEV void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
DEV void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
DEV void tma_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
DEV void mbar_wait(uint64_t* bar, uint32_t phase) {
    asm volatile("{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}"
                 ::"r"(smem_u32(bar)), "r"(phase) : "memory");
}

template <bool GEO>
__global__ void __launch_bounds__(256, 3) k_ntt_pass2(const PassArgs a) {
    extern __shared__ uint4 sh[];
    __shared__ uint64_t bar;
    const uint32_t M = 1u << a.logm, G = 1u << a.log_g, total = M << a.log_g, Q = M >> 2;
    uint4* dlo = sh; uint4* dhi = sh + total; uint4* tlo = sh + 2 * total; uint4* thi = tlo + M;
    const uint32_t tid = threadIdx.x;                  // blockDim.x == G * Q
    const uint32_t tiles_per_outer = a.inner_cnt >> a.log_g;
    const uint32_t bx = blockIdx.x + a.block0;
    const uint32_t outer = bx / tiles_per_outer, tile = bx % tiles_per_outer;
    const uint32_t inner0 = tile << a.log_g;
    const Fr* src = a.src + (size_t)blockIdx.y * a.src_pstride;
    Fr* dst = a.dst + (size_t)blockIdx.y * a.dst_pstride;
    const uint64_t slice_mask = (1ull << a.log_slice) - 1ull;
    const uint64_t in_base = (uint64_t)outer * a.in_outer_s + (uint64_t)inner0 * a.in_inner_s;
    const uint64_t out_base = (uint64_t)outer * a.out_outer_s + (uint64_t)inner0 * a.out_inner_s;

    if (tid == 0) mbar_init(&bar, 1);
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&bar, M * 32);
        tma_bulk_g2s(tlo, a.tw_staged, M * 16, &bar);
        tma_bulk_g2s(thi, a.tw_staged + M, M * 16, &bar);
    }

    int s = (int)a.logm - 1;
    bool first = true, tw_ready = false;
    while (s >= 0) {
        const bool two = !(first && (a.logm & 1u));            // odd log M: the first round is a single stage
        const int s_next = two ? s - 2 : s - 1;
        const bool last = s_next < 0;
        // thread -> (line g, quad t): g fastest where the global side is contiguous in g, t fastest otherwise
        uint32_t g, t;
        const bool g_fast = last || (first && !a.in_r_fast);
        if (g_fast) { g = tid & (G - 1); t = tid >> a.log_g; } else { t = tid & (Q - 1); g = tid >> (a.logm - 2); }
        const uint32_t q = 1u << (s - 1), p = t & (q - 1), blk = t >> (s - 1);
        const uint32_t base = (blk << (s + 1)) + p;
        Fr x[4];
        const bool sparse = first && a.first && a.n_in < ((uint64_t)M * a.inner_cnt);      // only the first round of a padded pass 1
        if (first) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint64_t idx = in_base + (uint64_t)g * a.in_inner_s + (uint64_t)(base + j * q) * a.in_rs;
                x[j] = fp_zero<FrTag>();
                if (idx < a.n_in) {
                    x[j] = fp_load(a.peer_on ? a.src_peers[idx >> a.log_slice] + (idx & slice_mask) : src + idx);
                    if (a.first) {
                        if constexpr (GEO) x[j] = x[j] * geo_power(a.pre, idx);
                        else if (a.pre.mode == 1) x[j] = x[j] * a.pre.c[0];
                        else if (a.pre.mode == 3) { uint32_t m3 = (uint32_t)(idx % 3); if (m3) x[j] = x[j] * a.pre.c[m3]; }
                    }
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) x[j] = sh_get(dlo, dhi, (g << a.logm) + base + j * q);
        }
        if (!tw_ready) { mbar_wait(&bar, 0); tw_ready = true; }
        // stage s: pairs (0,2) and (1,3), twiddles T_s[p], T_s[p+q]
        {
            const uint32_t o = (1u << s) - 1u;
            Fr u0 = x[0] + x[2], u2 = x[0] - x[2], u1 = x[1] + x[3], u3 = x[1] - x[3];
            if (s > 0) {
                // zero-padded inputs (coeff_to_extended: n of 2^ext_k coefficients): most first-round operands are zero,
                // and whole warps agree on which, so the multiplications are skipped without divergence
                if (p && !(sparse && fp_is_zero(u2))) u2 = u2 * sh_get(tlo, thi, o + p);
                if (!(sparse && fp_is_zero(u3))) u3 = u3 * sh_get(tlo, thi, o + p + q);
            }
            x[0] = u0; x[1] = u1; x[2] = u2; x[3] = u3;
        }
        if (two) {     // stage s-1: pairs (0,1) and (2,3), twiddle T_{s-1}[p]
            const uint32_t o = (1u << (s - 1)) - 1u;
            Fr v0 = x[0] + x[1], v1 = x[0] - x[1], v2 = x[2] + x[3], v3 = x[2] - x[3];
            if (s - 1 > 0 && p) {
                Fr w = sh_get(tlo, thi, o + p);
                if (!(sparse && fp_is_zero(v1))) v1 = v1 * w;
                if (!(sparse && fp_is_zero(v3))) v3 = v3 * w;
            }
            x[0] = v0; x[1] = v1; x[2] = v2; x[3] = v3;
        }
        if (!last) {
#pragma unroll
            for (int j = 0; j < 4; ++j) sh_put(dlo, dhi, (g << a.logm) + base + j * q, x[j]);     // in place: a quad is owned by one thread per round
            __syncthreads();
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t pos = base + j * q;
                const uint32_t rp = __brev(pos) >> (32 - a.logm);
                Fr v = x[j];
                if (a.tw_on) {
                    const uint64_t i_rest = a.rest_is_inner ? (uint64_t)(inner0 + g) : 0;
                    const uint64_t ex = a.tw_mul * (uint64_t)rp * i_rest;
                    if (ex) {
                        if (a.t_full) v = v * fp_load(a.t_full + ex);
                        else {
                            const uint32_t elo = (uint32_t)(ex & ((1ull << a.lo_bits) - 1)), ehi = (uint32_t)(ex >> a.lo_bits);
                            Fr w = fp_load(a.t_lo + elo);
                            if (ehi) w = w * fp_load(a.t_hi + ehi);
                            v = v * w;
                        }
                    }
                }
                const uint64_t idx = out_base + (uint64_t)g * a.out_inner_s + (uint64_t)rp * a.out_rs;
                if (a.last) {
                    if (a.post.mode == 1) v = v * a.post.c[0];
                    else if (a.post.mode == 3) v = v * a.post.c[(uint32_t)(idx % 3)];
                }
                fp_store(a.peer_on ? a.dst_peers[idx >> a.log_slice] + (idx & slice_mask) : dst + idx, v);
            }
        }
        first = false;
        s = s_next;
    }
}

// staged twiddles for one pass: entry (2^s - 1 + p) = w^(p << (logm - 1 - s)), written planar ([lo plane M][hi plane M])
__global__ void k_stage_twiddles(Fr w, uint32_t logm, uint4* __restrict__ out) {
    const uint32_t M = 1u << logm, idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M) return;
    Fr v = fp_zero<FrTag>();
    if (idx + 1 < M) {
        const uint32_t s = 31 - __clz(idx + 1), p = idx + 1 - (1u << s);
        v = fp_pow_u64(w, (uint64_t)p << (logm - 1 - s));
    }
    out[idx] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    out[M + idx] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}
// out[i] = base^i with one pow per 32-element run
__global__ void k_powers_run(Fr base, uint64_t count, Fr* __restrict__ out) {
    const uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 32;
    if (i0 >= count) return;
    Fr v = fp_pow_u64(base, i0);
    for (uint64_t i = i0; i < i0 + 32 && i < count; ++i) { fp_store(out + i, v); v = v * base; }
}

// out[i] = base^i  (i < count); twiddle-table builder
__global__ void k_powers(Fr base, uint32_t count, Fr* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) fp_store(out + i, fp_pow_u64(base, (uint64_t)i));
}

static void choose_passes(uint32_t log_n, int* npass, int logm[3]) {
    logm[0] = logm[1] = logm[2] = 0;
    if (log_n <= 10) { *npass = 1; logm[0] = (int)log_n; return; }
    if (log_n <= 20) { *npass = 2; logm[0] = (int)(log_n + 1) / 2; logm[1] = (int)log_n - logm[0]; return; }
    *npass = 3;
    logm[0] = (int)(log_n + 2) / 3; logm[1] = (int)(log_n - logm[0] + 1) / 2; logm[2] = (int)log_n - logm[0] - logm[1];
}
int ntt_launches_per_run(uint32_t log_n) { int np, lm[3]; choose_passes(log_n, &np, lm); return np; }

uint32_t geo_lo_bits(uint32_t log_n) { return (log_n + 1) / 2; }
size_t geo_table_len(uint32_t log_n) { return ((size_t)1 << geo_lo_bits(log_n)) + ((size_t)1 << (log_n - geo_lo_bits(log_n))); }
void geo_table_fill(const Fr& c, uint32_t log_n, Fr* out) {
    const uint32_t b = geo_lo_bits(log_n);
    const size_t nlo = (size_t)1 << b, nhi = (size_t)1 << (log_n - b);
    Fr v = fp_one<FrTag>();
    for (size_t i = 0; i < nlo; ++i) { out[i] = v; v = v * c; }          // v = c^(2^b) on exit
    Fr w = fp_one<FrTag>();
    for (size_t i = 0; i < nhi; ++i) { out[nlo + i] = w; w = w * v; }
}

static Fr host_pow(const Fr& b, uint64_t e) { return fp_pow_u64(b, e); }

NttPlan* NttContext::get(uint32_t log_n, const Fr& omega, cudaStream_t st) {
    for (NttPlan* p : plans) if (p->log_n == log_n && fp_eq(p->omega, omega)) return p;
    NttPlan* p = new NttPlan();
    p->log_n = log_n; p->omega = omega;
    choose_passes(log_n, &p->npass, p->logm);
    const uint64_t N = 1ull << log_n;
    for (int i = 0; i < p->npass; ++i) {
        const uint32_t M = 1u << p->logm[i], cnt = M > 1 ? M / 2 : 1;
        if (cudaMalloc(&p->d_tw[i], sizeof(Fr) * cnt) != cudaSuccess) { set_error("ntt plan: cudaMalloc failed"); delete p; return nullptr; }
        k_powers<<<div_up(cnt, 128), 128, 0, st>>>(host_pow(omega, N / M), cnt, p->d_tw[i]);
    }
    p->lo_bits = (log_n + 1) / 2;
    const uint32_t nlo = 1u << p->lo_bits, nhi = (uint32_t)(N >> p->lo_bits);
    if (cudaMalloc(&p->d_lo, sizeof(Fr) * nlo) != cudaSuccess || cudaMalloc(&p->d_hi, sizeof(Fr) * (nhi ? nhi : 1)) != cudaSuccess) {
        set_error("ntt plan: cudaMalloc failed"); delete p; return nullptr;
    }
    for (int i = 0; i < p->npass; ++i) {
        const uint32_t M = 1u << p->logm[i];
        if (cudaMalloc(&p->d_staged[i], sizeof(uint4) * 2 * M) != cudaSuccess) { set_error("ntt plan: cudaMalloc failed"); delete p; return nullptr; }
        k_stage_twiddles<<<div_up(M, 128), 128, 0, st>>>(host_pow(omega, N / M), (uint32_t)p->logm[i], p->d_staged[i]);
    }
    if (p->npass > 1 && log_n <= 25) {        // full single-multiply twiddle table (N * 32 B; falls back to the two-level table if it does not fit)
        if (cudaMalloc(&p->d_full, sizeof(Fr) * N) != cudaSuccess) { cudaGetLastError(); p->d_full = nullptr; }
        else k_powers_run<<<div_up(div_up(N, 32), 128), 128, 0, st>>>(omega, N, p->d_full);
    }
    k_powers<<<div_up(nlo, 128), 128, 0, st>>>(omega, nlo, p->d_lo);
    k_powers<<<div_up(nhi ? nhi : 1, 128), 128, 0, st>>>(host_pow(omega, 1ull << p->lo_bits), nhi ? nhi : 1, p->d_hi);
    if (cudaGetLastError() != cudaSuccess) { set_error("ntt plan: table kernel launch failed"); delete p; return nullptr; }
    plans.push_back(p);
    return p;
}
void NttContext::release() {
    for (NttPlan* p : plans) {
        for (int i = 0; i < 3; ++i) { if (p->d_tw[i]) cudaFree(p->d_tw[i]); if (p->d_staged[i]) cudaFree(p->d_staged[i]); }
        if (p->d_full) cudaFree(p->d_full);
        if (p->d_lo) cudaFree(p->d_lo);
        if (p->d_hi) cudaFree(p->d_hi);
        delete p;
    }
    plans.clear();
}

static int launch_pass_v1(PassArgs& a, uint64_t lines, int batch, cudaStream_t st);

// v2 launch geometry: G lines per CTA chosen so that a CTA holds 1024 elements (256 threads, one quad each; 3 CTAs per SM).
// Returns false when the pass has to take the v1 kernel (tiny passes).
static bool plan_pass_v2(PassArgs& a, uint64_t lines, int batch, uint32_t* threads, size_t* smem) {
    const Config& cfg = config();
    if (a.logm < 2 || cfg.ntt_v1) return false;
    uint32_t log_g = a.logm >= 10 ? 0 : 10 - a.logm;
    if (cfg.ntt_logg >= 0) log_g = (uint32_t)cfg.ntt_logg;
    while (log_g > 0 && ((1u << log_g) > a.inner_cnt || (lines >> log_g) * (uint64_t)batch < 296)) --log_g;
    while (log_g > 0 && (a.logm + log_g > 10)) --log_g;
    if (a.logm + log_g < 7) return false;       // fewer than 32 quads: not worth a CTA
    a.log_g = log_g;
    *threads = 1u << (a.logm + log_g - 2);
    *smem = (((size_t)1 << (a.logm + log_g)) + ((size_t)1 << a.logm)) * 32;
    return true;
}
static int launch_pass(PassArgs& a, uint64_t lines, int batch, cudaStream_t st) {
    uint32_t threads; size_t smem;
    if (!plan_pass_v2(a, lines, batch, &threads, &smem)) return launch_pass_v1(a, lines, batch, st);
    B200_CHECK(threads <= 256 && smem <= 200 * 1024, -1, "ntt: pass of 2^%u does not fit a CTA", a.logm);
    auto kern = a.pre.mode == NTT_SCALE_GEOMETRIC ? k_ntt_pass2<true> : k_ntt_pass2<false>;
    B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));     // per device, idempotent
    dim3 grid((unsigned)(lines >> a.log_g), (unsigned)batch);
    kern<<<grid, threads, smem, st>>>(a);
    B200_CUDA(cudaGetLastError());
    return 0;
}

static int launch_pass_v1(PassArgs& a, uint64_t lines, int batch, cudaStream_t st) {
    // lines per CTA: largest G in {4,2,1} that still yields >= 2 CTAs per SM (and fits shared memory)
    const Config& cfg = config();
    uint32_t log_g = 2;
    while (log_g > 0 && ((1u << log_g) > a.inner_cnt || (lines >> log_g) * (uint64_t)batch < 296)) --log_g;
    while (log_g > 0 && (((size_t)1 << (a.logm + log_g)) + ((size_t)1 << a.logm) / 2) * 32 > 200 * 1024) --log_g;
    if (cfg.ntt_logg >= 0) { uint32_t v = (uint32_t)cfg.ntt_logg; while (v > 0 && (1u << v) > a.inner_cnt) --v; log_g = v; }
    a.log_g = log_g;
    const size_t smem = (((size_t)1 << (a.logm + log_g)) + (((size_t)1 << a.logm) >> 1)) * 32;
    const uint32_t nbf = (1u << (a.logm + log_g)) >> 1;
    uint32_t threads = nbf < 32 ? 32 : (nbf > 1024 ? 1024 : nbf);
    if (cfg.ntt_threads >= 32 && cfg.ntt_threads <= 1024 && (uint32_t)cfg.ntt_threads < threads) threads = (uint32_t)cfg.ntt_threads;
    auto kern = a.pre.mode == NTT_SCALE_GEOMETRIC ? k_ntt_pass<true> : k_ntt_pass<false>;
    B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));     // per device, idempotent
    dim3 grid((unsigned)(lines >> log_g), (unsigned)batch);
    kern<<<grid, threads, smem, st>>>(a);
    B200_CUDA(cudaGetLastError());
    return 0;
}

// Geometry of pass `idx` of a plan: which buffer it reads / writes (0 = source, 1 = scratch, 2 = destination), its strides,
// inter-pass twiddle and how many lines it transforms.  Shared by the single-device and the sharded drivers.
struct PassRole { int in_buf, out_buf; uint64_t lines; };
static PassRole fill_pass(const NttPlan* p, int idx, uint64_t n_in, PassArgs& a) {
    const uint64_t N1 = 1ull << p->logm[0], N2 = 1ull << p->logm[1], N3 = 1ull << p->logm[2], N23 = N2 * N3;
    a.t_lo = p->d_lo; a.t_hi = p->d_hi; a.lo_bits = p->lo_bits; a.t_full = config().ntt_nofull ? nullptr : p->d_full;
    a.tw_m = p->d_tw[idx]; a.tw_staged = p->d_staged[idx]; a.logm = p->logm[idx];
    a.in_outer_s = a.out_outer_s = 0; a.tw_on = 0; a.rest_is_inner = 0; a.tw_mul = 0;
    PassRole r{0, 2, 1};
    if (p->npass == 1) {
        a.inner_cnt = 1; a.in_r_fast = 1; a.in_rs = 1; a.in_inner_s = 0; a.out_rs = 1; a.out_inner_s = 0; a.n_in = n_in; a.first = a.last = 1;
        return r;
    }
    if (p->npass == 2) {
        if (idx == 0) {      // columns i2 (stride 1), transform over i1 (stride N2); twiddle omega^(j1 * i2)
            a.inner_cnt = (uint32_t)N2; a.in_r_fast = 0; a.in_rs = N2; a.in_inner_s = 1; a.out_rs = N2; a.out_inner_s = 1; a.n_in = n_in; a.first = 1; a.last = 0;
            a.tw_on = 1; a.rest_is_inner = 1; a.tw_mul = 1;
            r = PassRole{0, 1, N2};
        } else {             // rows j1 (stride N2), transform over i2 (stride 1); X[j1 + N1*j2]
            a.inner_cnt = (uint32_t)N1; a.in_r_fast = 1; a.in_rs = 1; a.in_inner_s = N2; a.out_rs = N1; a.out_inner_s = 1; a.n_in = ~0ull; a.first = 0; a.last = 1;
            r = PassRole{1, 2, N1};
        }
        return r;
    }
    // three passes: i = i1*N2*N3 + i2*N3 + i3  ->  j = j1 + N1*j2 + N1*N2*j3
    if (idx == 0) {
        a.inner_cnt = (uint32_t)N23; a.in_r_fast = 0; a.in_rs = N23; a.in_inner_s = 1; a.out_rs = N23; a.out_inner_s = 1; a.n_in = n_in; a.first = 1; a.last = 0;
        a.tw_on = 1; a.rest_is_inner = 1; a.tw_mul = 1;
        r = PassRole{0, 1, N23};
    } else if (idx == 1) {   // in place on scratch: outer j1 (stride N23), inner i3 (stride 1), transform over i2 (stride N3); twiddle omega^(N1*j2*i3)
        a.inner_cnt = (uint32_t)N3; a.in_r_fast = 0; a.in_rs = N3; a.in_inner_s = 1; a.in_outer_s = N23; a.out_rs = N3; a.out_inner_s = 1; a.out_outer_s = N23;
        a.n_in = ~0ull; a.first = 0; a.last = 0; a.tw_on = 1; a.rest_is_inner = 1; a.tw_mul = N1;
        r = PassRole{1, 1, N1 * N3};
    } else {                 // outer j2 (stride N3), inner j1 (stride N23), transform over i3 (stride 1)
        a.inner_cnt = (uint32_t)N1; a.in_r_fast = 1; a.in_rs = 1; a.in_inner_s = N23; a.in_outer_s = N3; a.out_rs = N1 * N2; a.out_inner_s = 1; a.out_outer_s = N1;
        a.n_in = ~0ull; a.first = 0; a.last = 1;
        r = PassRole{1, 2, N1 * N2};
    }
    return r;
}

int ntt_run(NttPlan* p, const Fr* d_src, size_t src_stride, size_t n_in, Fr* d_tmp, size_t tmp_stride, Fr* d_dst, size_t dst_stride,
            uint32_t log_n, const Fr& omega, const NttScale& pre, const NttScale& post, int batch, cudaStream_t st) {
    B200_CHECK(log_n >= 1 && log_n <= 28, -1, "ntt: log_n = %u out of range [1, 28]", log_n);
    B200_CHECK(batch > 0 && batch <= 65535, -1, "ntt: batch %d out of range", batch);
    const uint64_t N = 1ull << log_n;
    B200_CHECK(n_in <= N, -1, "ntt: n_in %zu > N", n_in);
    B200_CHECK(p && p->log_n == log_n && fp_eq(p->omega, omega), -1, "ntt: plan does not match (log_n, omega)");
    B200_CHECK(post.mode != NTT_SCALE_GEOMETRIC && (pre.mode != NTT_SCALE_GEOMETRIC || (pre.lo && pre.hi && pre.lo_bits <= log_n)), -1,
               "ntt: the geometric scale is a pre-scale with both power tables");
    ProfScope ps(PROF_NTT, st);
    PassArgs a;
    memset(&a, 0, sizeof a);
    a.pre = pre; a.post = post;
    const Fr* bufs[3] = {d_src, d_tmp, d_dst};
    const size_t strides[3] = {src_stride, tmp_stride, dst_stride};
    for (int idx = 0; idx < p->npass; ++idx) {
        const PassRole r = fill_pass(p, idx, n_in, a);
        a.src = bufs[r.in_buf]; a.src_pstride = strides[r.in_buf];
        a.dst = const_cast<Fr*>(bufs[r.out_buf]); a.dst_pstride = strides[r.out_buf];
        if (int rc = launch_pass(a, r.lines, batch, st)) return rc;
    }
    return 0;
}

// One transform of 2^log_n elements split across ndev devices in contiguous natural-order slices (slice g on device g, in and
// out).  Every pass runs on all devices at once, device g taking the g-th share of the pass's CTAs; loads and stores go through
// the peer tables (NVLink loads / stores inside the butterfly kernel), so the all-to-all exchanges of the six-step scheme never
// exist as separate copies.  Between passes every stream waits for every other device's pass (events).  plans[g], st[g], ev[g]
// belong to device dev_ids[g]; the caller has enabled peer access.  dst may alias src; tmp must not alias either.
int ntt_run_sharded(NttPlan* const* plans, int ndev, const int* dev_ids, const Fr* const* src, Fr* const* tmp, Fr* const* dst, uint32_t log_n, const Fr& omega,
                    const NttScale& pre, const NttScale& post, uint64_t n_in, cudaStream_t* st, cudaEvent_t* ev) {
    B200_CHECK(ndev >= 2 && ndev <= 8 && (ndev & (ndev - 1)) == 0, -1, "sharded ntt: device count %d must be 2, 4 or 8", ndev);
    uint32_t log_d = 0;
    while ((1 << log_d) < ndev) ++log_d;
    B200_CHECK(log_n >= 12 && log_n <= 28, -1, "sharded ntt: log_n = %u out of range [12, 28]", log_n);
    const uint64_t N = 1ull << log_n;
    B200_CHECK(n_in <= N, -1, "sharded ntt: n_in > N");
    B200_CHECK(pre.mode != NTT_SCALE_GEOMETRIC && post.mode != NTT_SCALE_GEOMETRIC, -1, "sharded ntt: the geometric pre-scale is not supported");
    for (int g = 0; g < ndev; ++g) B200_CHECK(plans[g] && plans[g]->log_n == log_n && fp_eq(plans[g]->omega, omega), -1, "sharded ntt: plan %d does not match", g);
    int cur = 0;
    cudaGetDevice(&cur);
    const Fr* const* bufs_r[3] = {src, tmp, dst};
    for (int idx = 0; idx < plans[0]->npass; ++idx) {
        for (int g = 0; g < ndev; ++g) {
            PassArgs a;
            memset(&a, 0, sizeof a);
            a.pre = pre; a.post = post;
            const PassRole r = fill_pass(plans[g], idx, n_in, a);
            uint32_t threads; size_t smem;
            if (!plan_pass_v2(a, r.lines, 1, &threads, &smem) || threads > 256 || smem > 200 * 1024) { cudaSetDevice(cur); set_error("sharded ntt: pass %d of 2^%u is too small to shard", idx, log_n); return -1; }
            const uint64_t blocks = r.lines >> a.log_g;
            if (blocks % (uint64_t)ndev) { cudaSetDevice(cur); set_error("sharded ntt: %llu CTAs do not divide over %d devices", (unsigned long long)blocks, ndev); return -1; }
            a.peer_on = 1; a.log_slice = log_n - log_d; a.block0 = (uint32_t)(blocks / ndev * g);
            for (int h = 0; h < ndev; ++h) { a.src_peers[h] = bufs_r[r.in_buf][h]; a.dst_peers[h] = const_cast<Fr*>(bufs_r[r.out_buf][h]); }
            B200_CUDA(cudaSetDevice(dev_ids[g]));
            B200_CUDA(cudaFuncSetAttribute(k_ntt_pass2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            k_ntt_pass2<false><<<dim3((unsigned)(blocks / ndev), 1), threads, smem, st[g]>>>(a);
            B200_CUDA(cudaGetLastError());
            B200_CUDA(cudaEventRecord(ev[g], st[g]));
        }
        for (int g = 0; g < ndev; ++g) {
            B200_CUDA(cudaSetDevice(dev_ids[g]));
            for (int h = 0; h < ndev; ++h) if (h != g) B200_CUDA(cudaStreamWaitEvent(st[g], ev[h], 0));
        }
    }
    B200_CUDA(cudaSetDevice(cur));
    return 0;
}

}  // namespace b200
