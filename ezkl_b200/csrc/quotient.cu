// quotient.cu — device side of halo2's `evaluate_h` (UPSTREAM plonk/evaluation.rs: Evaluator::evaluate_h / GraphEvaluator),
// the quotient-numerator stage of create_proof (SURVEY.md §3.1 stage 6, entered from /root/reference/src/pfsys/mod.rs:456).
//
// halo2 compiles every gate, permutation and lookup constraint into a straight-line program of field operations over
// "value sources" (column cosets at a rotation, constants, challenges, earlier intermediates; its Horner calculation is a chain
// of multiply-adds) and runs it once per row of the extended domain.  This kernel is that interpreter: one thread per extended
// row, uniform control flow.  The whole program — instructions, resolved column loads (pointer + cyclic offset) and constants —
// is staged ONCE per CTA into shared memory; intermediates live in a per-thread slot file of 32 / 64 / 128 / 256 entries
// (local memory, sized to the program), and a value consumed only by the next instruction never touches it (PREV operand,
// NOSTORE flag).  The Rust side lowers its GraphEvaluator calculations to QInstr (include/ezkl_b200.h: b200_instr);
// l0 / l_last / l_active_row, the identity coset X and previous partial sums are ordinary columns, y / beta / gamma / theta and the
// phase challenges are constants.  HBM traffic per row: 32 B per distinct column + 32 B store when a CTA's rows are contiguous
// (rotated re-reads of a column hit L1 / L2); arithmetic is bound by the same multiply ceiling as every other kernel here.
#include <vector>
#include "quotient.cuh"

namespace b200 {

struct QLoadDev { const Fr* col; uint32_t offset, pad; };      // 16 B: column pointer resolved on the host

// PARTS: one coset part of the extended domain (quotient_eval_part_run).  Row idx < 2^k of part r loads column element
// ((idx + offset) & mask) << pad, where pad = 0 for a part column and log2 d for a full extended column whose pointer is already
// advanced by r, and stores its result at out[idx << out_shift] with out advanced by r.  A separate instantiation: the
// whole-domain kernels keep their code.
template <int NSLOT, bool PARTS>
__global__ void __launch_bounds__(128) k_quotient_eval(const uint4* __restrict__ blob, uint32_t blob_u4, uint32_t o_loads_u4, uint32_t o_consts_u4, uint32_t mask,
                                                        uint32_t n_instr, Fr* __restrict__ out, uint32_t out_shift) {
    extern __shared__ uint4 sh[];
    for (uint32_t i = threadIdx.x; i < blob_u4; i += blockDim.x) sh[i] = blob[i];
    __syncthreads();
    const QInstr* prog = reinterpret_cast<const QInstr*>(sh);
    const QLoadDev* loads = reinterpret_cast<const QLoadDev*>(sh + o_loads_u4);
    const Fr* consts = reinterpret_cast<const Fr*>(sh + o_consts_u4);
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx > mask) return;
    Fr slots[NSLOT];
    Fr prev = fp_zero<FrTag>();
    auto fetch = [&](uint32_t s) -> Fr {
        const uint32_t k = s >> 30, i = s & 0x3fffffffu;
        if (k == QSRC_PREV) return prev;
        if (k == QSRC_SLOT) return slots[i & (NSLOT - 1)];
        if (k == QSRC_CONST) return fp_load(consts + i);
        const QLoadDev l = loads[i];
        if constexpr (PARTS) return fp_load(l.col + (((idx + l.offset) & mask) << l.pad));
        else return fp_load(l.col + ((idx + l.offset) & mask));
    };
#pragma unroll 1
    for (uint32_t pc = 0; pc < n_instr; ++pc) {
        const QInstr in = prog[pc];
        const uint32_t op = in.op_dst & 0xff;
        const Fr x = fetch(in.a);
        Fr r;
        if (op <= QOP_MUL) {
            const Fr y = fetch(in.b);
            r = op == QOP_ADD ? x + y : (op == QOP_SUB ? x - y : x * y);
        } else if (op == QOP_MULADD) {
            const Fr y = fetch(in.b), z = fetch(in.c);
            r = x * y + z;
        } else if (op == QOP_NEG) r = fp_neg(x);
        else if (op == QOP_DOUBLE) r = fp_dbl(x);
        else if (op == QOP_SQUARE) r = fp_sqr(x);
        else r = x;
        if (!(in.op_dst & Q_NOSTORE)) slots[(in.op_dst >> 8) & (NSLOT - 1)] = r;
        prev = r;
    }
    // the row's result is the last instruction's (zero for an empty program)
    if constexpr (PARTS) fp_store(out + ((size_t)idx << out_shift), prev);
    else fp_store(out + idx, prev);
}

// shared by both entry points: validates the program against n_cols columns and a row domain of 2^log_rows, stages it, launches.
// col_shift == nullptr: the whole extended domain (offsets < 2^log_rows); otherwise one coset part (out_shift = log2 d).
static int quotient_launch(const Fr* const* h_col_ptrs, const uint32_t* col_shift, size_t n_cols, uint32_t log_rows, const QLoad* h_loads, size_t n_loads,
                           const Fr* h_consts, size_t n_consts, const QInstr* h_prog, size_t n_instr, Fr* d_out, uint32_t out_shift, QuotientWorkspace& ws,
                           cudaStream_t st) {
    B200_CHECK(log_rows >= 1 && log_rows <= 28, -1, "quotient_eval: ext_k %u out of range", log_rows);
    B200_CHECK(n_instr < (1u << 24) && n_loads < (1u << 30) && n_consts < (1u << 30), -1, "quotient_eval: program too large");
    const uint32_t N = 1u << log_rows;
    // validate the program on the host so the kernel can index without checks
    for (size_t i = 0; i < n_loads; ++i) B200_CHECK(h_loads[i].column < n_cols && h_loads[i].offset < N, -1, "quotient_eval: load %zu out of range", i);
    uint32_t max_slot = 0;
    for (size_t pc = 0; pc < n_instr; ++pc) {
        const uint32_t op = h_prog[pc].op_dst & 0xff, dst = (h_prog[pc].op_dst >> 8) & 0xffff;
        B200_CHECK(op <= QOP_MULADD && dst < (uint32_t)Q_MAX_SLOTS, -1, "quotient_eval: instruction %zu: bad op %u / slot %u", pc, op, dst);
        if (!(h_prog[pc].op_dst & Q_NOSTORE) && dst > max_slot) max_slot = dst;
        const uint32_t srcs[3] = {h_prog[pc].a, h_prog[pc].b, h_prog[pc].c};
        const int nsrc = op == QOP_MULADD ? 3 : (op <= QOP_MUL ? 2 : 1);
        for (int s = 0; s < nsrc; ++s) {
            const uint32_t k = srcs[s] >> 30, i = srcs[s] & 0x3fffffffu;
            B200_CHECK((k == QSRC_SLOT && i < (uint32_t)Q_MAX_SLOTS) || (k == QSRC_CONST && i < n_consts) || (k == QSRC_LOAD && i < n_loads) || (k == QSRC_PREV && pc > 0), -1,
                       "quotient_eval: instruction %zu: bad operand", pc);
            if (k == QSRC_SLOT && i > max_slot) max_slot = i;
        }
    }
    // one blob, staged to the device once and copied to shared memory by every CTA: [prog | loads | consts]
    const size_t o_loads = sizeof(QInstr) * n_instr, o_consts = o_loads + sizeof(QLoadDev) * n_loads, total = o_consts + sizeof(Fr) * n_consts + 16;
    B200_CHECK(total <= 160 * 1024, -1, "quotient_eval: program of %zu bytes exceeds the 160 KB shared-memory stage; split it into partial sums", total);
    std::vector<uint8_t> blob(total, 0);
    if (n_instr) memcpy(blob.data(), h_prog, sizeof(QInstr) * n_instr);
    for (size_t i = 0; i < n_loads; ++i) {
        QLoadDev l; l.col = h_col_ptrs[h_loads[i].column]; l.offset = h_loads[i].offset; l.pad = col_shift ? col_shift[h_loads[i].column] : 0;
        memcpy(blob.data() + o_loads + sizeof(QLoadDev) * i, &l, sizeof l);
    }
    if (n_consts) memcpy(blob.data() + o_consts, h_consts, sizeof(Fr) * n_consts);
    uint8_t* d = reinterpret_cast<uint8_t*>(ws.ring.push(blob.data(), total, st));
    if (!d) {
        if (ws.prog.ensure(total)) return -2;
        B200_CUDA(cudaMemcpyAsync(ws.prog.p, blob.data(), total, cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaStreamSynchronize(st));      // blob is a stack temporary
        d = ws.prog.as<uint8_t>();
    }
    const uint32_t blob_u4 = (uint32_t)((total + 15) / 16);
    const size_t smem = (size_t)blob_u4 * 16;
    const dim3 grid(div_up(N, 128));
    ProfScope ps(PROF_QUOTIENT, st);
#define B200_QLAUNCH(NS, PARTS)                                                                                                       \
    do {                                                                                                                              \
        B200_CUDA(cudaFuncSetAttribute(k_quotient_eval<NS, PARTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024 + 64));     \
        k_quotient_eval<NS, PARTS><<<grid, 128, smem, st>>>(reinterpret_cast<const uint4*>(d), blob_u4, (uint32_t)(o_loads / 16), (uint32_t)(o_consts / 16), \
                                                            N - 1, (uint32_t)n_instr, d_out, out_shift);                                \
    } while (0)
    if (col_shift) {
        if (max_slot < 32) B200_QLAUNCH(32, true);
        else if (max_slot < 64) B200_QLAUNCH(64, true);
        else if (max_slot < 128) B200_QLAUNCH(128, true);
        else B200_QLAUNCH(256, true);
    } else {
        if (max_slot < 32) B200_QLAUNCH(32, false);
        else if (max_slot < 64) B200_QLAUNCH(64, false);
        else if (max_slot < 128) B200_QLAUNCH(128, false);
        else B200_QLAUNCH(256, false);
    }
#undef B200_QLAUNCH
    B200_CUDA(cudaGetLastError());
    return 0;
}

int quotient_eval_run(const Fr* const* h_col_ptrs, size_t n_cols, uint32_t ext_k, const QLoad* h_loads, size_t n_loads, const Fr* h_consts, size_t n_consts,
                      const QInstr* h_prog, size_t n_instr, Fr* d_out, QuotientWorkspace& ws, cudaStream_t st) {
    return quotient_launch(h_col_ptrs, nullptr, n_cols, ext_k, h_loads, n_loads, h_consts, n_consts, h_prog, n_instr, d_out, 0, ws, st);
}

int quotient_eval_part_run(const Fr* const* h_col_ptrs, const uint32_t* h_col_shift, size_t n_cols, uint32_t k, uint32_t log_d, const QLoad* h_loads, size_t n_loads,
                           const Fr* h_consts, size_t n_consts, const QInstr* h_prog, size_t n_instr, Fr* d_out, QuotientWorkspace& ws, cudaStream_t st) {
    B200_CHECK(h_col_shift || n_cols == 0, -1, "quotient_eval: part layout missing");
    for (size_t i = 0; i < n_cols; ++i) B200_CHECK(h_col_shift[i] == 0 || h_col_shift[i] == log_d, -1, "quotient_eval: column %zu: bad part stride", i);
    static const uint32_t no_cols = 0;
    return quotient_launch(h_col_ptrs, n_cols ? h_col_shift : &no_cols, n_cols, k, h_loads, n_loads, h_consts, n_consts, h_prog, n_instr, d_out, log_d, ws, st);
}

}  // namespace b200
