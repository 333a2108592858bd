// quotient.cuh — row-wise expression-program evaluator over extended cosets (the device side of evaluate_h).
#pragma once
#include "common.cuh"
#include "field.cuh"

namespace b200 {

// Operand encoding: bits 31..30 = kind (0 slot, 1 constant, 2 column load, 3 the previous instruction's result), bits 29..0 = index.
enum QSrcKind { QSRC_SLOT = 0, QSRC_CONST = 1, QSRC_LOAD = 2, QSRC_PREV = 3 };
enum QOp { QOP_ADD = 0, QOP_SUB = 1, QOP_MUL = 2, QOP_NEG = 3, QOP_DOUBLE = 4, QOP_SQUARE = 5, QOP_MOV = 6, QOP_MULADD = 7 };
static constexpr int Q_MAX_SLOTS = 256;
static constexpr uint32_t Q_NOSTORE = 0x80000000u;     // op_dst flag: the result is only read as PREV by the next instruction

struct QInstr { uint32_t op_dst; uint32_t a, b, c; };   // op_dst = op | (dst_slot << 8) | NOSTORE;  MULADD: a * b + c
struct QLoad { uint32_t column; uint32_t offset; };      // element offset already reduced mod 2^ext_k

struct QuotientWorkspace { DevBuf prog; StagingRing ring; };

// out[idx] = program(columns[c][(idx + offset) mod N], constants) for idx < N = 2^ext_k.  h_* are host arrays.
int quotient_eval_run(const Fr* const* h_col_ptrs /*device addresses*/, size_t n_cols, uint32_t ext_k, const QLoad* h_loads, size_t n_loads,
                      const Fr* h_consts, size_t n_consts, const QInstr* h_prog, size_t n_instr, Fr* d_out, QuotientWorkspace& ws, cudaStream_t st);
// One coset part r of the extended domain (d = 2^log_d parts of 2^k rows each): out[idx << log_d] = program(...) for idx < 2^k, where
// column c is read at ((idx + offset) mod 2^k) << h_col_shift[c].  h_col_shift[c] = 0: a part column (2^k values of that part);
// log_d: a full extended column whose device address is already advanced by r.  d_out is advanced by r.  Offsets are Rotation(rot) mod 2^k.
int quotient_eval_part_run(const Fr* const* h_col_ptrs, const uint32_t* h_col_shift, size_t n_cols, uint32_t k, uint32_t log_d, const QLoad* h_loads, size_t n_loads,
                           const Fr* h_consts, size_t n_consts, const QInstr* h_prog, size_t n_instr, Fr* d_out, QuotientWorkspace& ws, cudaStream_t st);

}  // namespace b200
