/*
 * ezkl_b200_parts.h — the extended domain one coset part at a time: evaluate_h for systems whose columns' full cosets do not fit
 * on one device together.
 *
 * The extended domain {zeta * w_N^j : j < N} (N = 2^ext_k, w_N = ext_omega, n = 2^k, d = N / n, w_n = w_N^d) is the union of d
 * cosets of the size-n subgroup: part r = {c_r * w_n^t : t < n} with c_r = zeta * w_N^r, and extended index j = t * d + r.
 *   - a coefficient-form column's values on part r are one size-n transform of p_i * c_r^i;
 *   - Rotation(rot), which is rot * d on the extended index, is rot inside a part, so every part is a self-contained size-n evaluate_h;
 *   - the vanishing polynomial is constant on a part: c_r^n - 1 (t_evaluations[r mod t_period] holds its inverse).
 * Written back to their interleaved positions, the parts' numerators are exactly b200_evaluate_h's numerator, and the same extended
 * inverse transform yields the same quotient coefficients: the output equals b200_evaluate_h's byte for byte wherever that fits.
 * (UNPINNED, from recollection of PSE-lineage halo2: Evaluator::evaluate_h looping over num_parts with
 * EvaluationDomain::coeff_to_extended_part and lagrange_vecs_to_extended; INTEGRATION.md §2.)
 *
 * Conventions are those of ezkl_b200.h: return 0 = ok, -1 bad argument, -2 CUDA failure, -3 not initialised, message via
 * b200_last_error(); the library guard is checked before anything else; `_dev` entries take device pointers and a cudaStream_t
 * (NULL = the calling thread's library stream) and do not synchronise.  In a multi-device process these entries run on ONE device:
 * a `_dev` entry on the device that owns its first device pointer (d_coeffs, or d_out for b200_evaluate_h_parts_dev), a host entry
 * on the calling thread's slot 0.
 */
#ifndef EZKL_B200_PARTS_H
#define EZKL_B200_PARTS_H

#include "ezkl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* out[p][t] = coeffs[p](zeta * ext_omega^part * w_n^t), t < 2^k, w_n = ext_omega^(2^(ext_k - k)): part `part` of coeff_to_extended, i.e.
 * coeff_to_extended(coeffs[p])[part :: 2^(ext_k - k)].  n_coeffs <= 2^k, part < 2^(ext_k - k), k >= 1. */
int b200_coeff_to_extended_part_batch(const b200_fr* const* coeffs, size_t batch, size_t n_coeffs, uint32_t k, uint32_t ext_k, uint32_t part,
                                      const b200_fr* ext_omega, const b200_fr* zeta, b200_fr* const* out);
/* device form: polynomial p at d_coeffs + p * src_stride (n_coeffs valid elements), its part at d_out + p * dst_stride (2^k elements);
 * d_tmp: 2^k * batch elements of scratch, as b200_ntt_dev takes. */
int b200_coeff_to_extended_part_dev(const void* d_coeffs, size_t src_stride, size_t n_coeffs, void* d_tmp, void* d_out, size_t dst_stride, uint32_t k,
                                    uint32_t ext_k, uint32_t part, const b200_fr* ext_omega, const b200_fr* zeta, size_t batch, void* stream);

/* b200_evaluate_h evaluated one coset part at a time: the same arguments and the same output.  t_evaluations == NULL: the numerator on the
 * extended domain in natural order; otherwise the quotient's 2^ext_k coefficients.  Column i is a coefficient column when
 * lengths[i] <= 2^k and an extended column (values on the whole extended domain) when lengths[i] == 2^ext_k; any other length is
 * rejected (-1).  t_period must divide 2^(ext_k - k).  The program gains one multiplication by the part's vanishing factor when
 * finishing, so it must fit the 160 KB stage with 48 bytes to spare.
 * Coefficient columns are uploaded once and stay resident across the parts; part r of an extended column is gathered from the
 * caller's buffer (stride 2^(ext_k - k)) through the pinned staging buffers, so an extended column never sits whole on the device.
 * Device memory: part buffers n_coeff_cols * 2^k * 32 B, plus the output and the transform scratch 2 * 2^ext_k * 32 B, plus the
 * resident coefficients (sum of their lengths * 32 B) and one part of every extended column (n_extended * 2^k * 32 B). */
int b200_evaluate_h_parts(const b200_fr* const* polys, const size_t* lengths, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_fr* ext_omega,
                          const b200_fr* zeta, const b200_col_ref* loads, size_t n_loads, const b200_fr* constants, size_t n_constants,
                          const b200_instr* program, size_t n_instr, const b200_fr* t_evaluations, uint32_t t_period, const b200_fr* ext_omega_inv,
                          const b200_fr* ext_ifft_divisor, b200_fr* out);
/* device form: d_polys is a host array of device addresses; coefficient and extended columns are read in place (an extended column at
 * stride 2^(ext_k - k) per part), the result goes to d_out (2^ext_k elements).  Device memory held by the library: part buffers
 * n_coeff_cols * 2^k * 32 B plus the transform scratch 2^ext_k * 32 B (the caller's d_out is the other 2^ext_k * 32 B). */
int b200_evaluate_h_parts_dev(const void* const* d_polys, const size_t* lengths, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_fr* ext_omega,
                              const b200_fr* zeta, const b200_col_ref* loads, size_t n_loads, const b200_fr* constants, size_t n_constants,
                              const b200_instr* program, size_t n_instr, const b200_fr* t_evaluations, uint32_t t_period, const b200_fr* ext_omega_inv,
                              const b200_fr* ext_ifft_divisor, void* d_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EZKL_B200_PARTS_H */
