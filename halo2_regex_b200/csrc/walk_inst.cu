// Instantiates walk_kernel and emit_kernel for one number of regex defs (compiled once per D with -DB2R_INST_D=<D>, in
// parallel).  With -DB2R_INST_CH=1 the same file instantiates the chunked-batch walk_kernel only (b2r_match_batch_chunked).
#include "emit.cuh"
#include "walk.cuh"

#ifndef B2R_INST_D
#error "compile with -DB2R_INST_D=<1..4>"
#endif
#ifndef B2R_INST_CH
#define B2R_INST_CH 0
#endif

namespace b2r {

template <int D, typename ST, int TM, int HM>
static int launch_walk_one(const WalkParams& p, size_t smem, int grid, int block, cudaStream_t st) {
    auto kern = walk_kernel<D, ST, TM, HM, (bool)B2R_INST_CH>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(walk_kernel): %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    kern<<<grid, block, smem, st>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("walk_kernel launch: %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    return B2R_OK;
}

template <int D, bool CH>
int launch_walk_d(const WalkParams& p, bool wide, size_t smem, int grid, int block, cudaStream_t st);

template <>
int launch_walk_d<B2R_INST_D, (bool)B2R_INST_CH>(const WalkParams& p, bool wide, size_t smem, int grid, int block, cudaStream_t st) {
    constexpr int D = B2R_INST_D;
    const uint32_t tm = p.table_mode;
    const bool shist = p.hist_mode == HIST_SMEM;
    if (wide) {   // 2-byte states: more than 255 states, the bins never fit in shared memory
        if (shist) { set_error("walk_kernel: shared-memory bins with 2-byte states"); return B2R_ERR_UNSUPPORTED; }
        switch (tm) {
            case TABLE_REPL: return launch_walk_one<D, uint16_t, TABLE_REPL, HIST_GLOBAL>(p, smem, grid, block, st);
            case TABLE_REPL16: return launch_walk_one<D, uint16_t, TABLE_REPL16, HIST_GLOBAL>(p, smem, grid, block, st);
            case TABLE_PLAIN: return launch_walk_one<D, uint16_t, TABLE_PLAIN, HIST_GLOBAL>(p, smem, grid, block, st);
            case TABLE_PLAIN16: return launch_walk_one<D, uint16_t, TABLE_PLAIN16, HIST_GLOBAL>(p, smem, grid, block, st);
            default: return launch_walk_one<D, uint16_t, TABLE_GLOBAL, HIST_GLOBAL>(p, smem, grid, block, st);
        }
    }
    if (tm == TABLE_GLOBAL) {
        if (shist) { set_error("walk_kernel: shared-memory bins with global tables"); return B2R_ERR_UNSUPPORTED; }
        return launch_walk_one<D, uint8_t, TABLE_GLOBAL, HIST_GLOBAL>(p, smem, grid, block, st);
    }
    if (tm == TABLE_REPL)
        return shist ? launch_walk_one<D, uint8_t, TABLE_REPL, HIST_SMEM>(p, smem, grid, block, st)
                     : launch_walk_one<D, uint8_t, TABLE_REPL, HIST_GLOBAL>(p, smem, grid, block, st);
    if (tm == TABLE_REPL16)
        return shist ? launch_walk_one<D, uint8_t, TABLE_REPL16, HIST_SMEM>(p, smem, grid, block, st)
                     : launch_walk_one<D, uint8_t, TABLE_REPL16, HIST_GLOBAL>(p, smem, grid, block, st);
    if (tm == TABLE_PLAIN16)
        return shist ? launch_walk_one<D, uint8_t, TABLE_PLAIN16, HIST_SMEM>(p, smem, grid, block, st)
                     : launch_walk_one<D, uint8_t, TABLE_PLAIN16, HIST_GLOBAL>(p, smem, grid, block, st);
    return shist ? launch_walk_one<D, uint8_t, TABLE_PLAIN, HIST_SMEM>(p, smem, grid, block, st)
                 : launch_walk_one<D, uint8_t, TABLE_PLAIN, HIST_GLOBAL>(p, smem, grid, block, st);
}

#if !B2R_INST_CH
template <int D>
int launch_emit_d(const WalkParams& p, bool wide, size_t smem, int grid, cudaStream_t st);

template <int D, typename ST>
static int launch_emit_one(const WalkParams& p, size_t smem, int grid, cudaStream_t st) {
    auto kern = emit_kernel<D, ST>;
    if (smem + EMIT_ZERO_BYTES > 48 * 1024) {   // + the static zero buffer: past 48 KB in all, the kernel has to opt in
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(emit_kernel): %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    }
    kern<<<grid, EMIT_THREADS, smem, st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("emit_kernel launch: %s", cudaGetErrorString(e)); return B2R_ERR_CUDA; }
    return B2R_OK;
}

template <>
int launch_emit_d<B2R_INST_D>(const WalkParams& p, bool wide, size_t smem, int grid, cudaStream_t st) {
    constexpr int D = B2R_INST_D;
    return wide ? launch_emit_one<D, uint16_t>(p, smem, grid, st) : launch_emit_one<D, uint8_t>(p, smem, grid, st);
}
#endif

}  // namespace b2r
