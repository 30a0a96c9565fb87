/*
 * emu_plans.cpp -- the product's FIR launch plans (stm32f7-rtlsdr_b200/csrc/plan.h) behind a C ABI, so
 * tests/test_gpu_plan_regimes.py can pin the shapes it runs to their regimes without a GPU.  TEST
 * INFRASTRUCTURE ONLY.  That test builds it into a temporary directory:
 *   g++ -O1 -std=c++17 -shared -fPIC -o libemu_plans.so emu_plans.cpp
 * (the spectrum plan is emu_plan_spectrum of emu_kernels.cpp)
 */
#include "cuda_emu.h"

#include "../../stm32f7-rtlsdr_b200/csrc/plan.h"

extern "C" {

/* the FP32 WBFM batch plan: out4 = n_tiles, total_chunks, tiles_per_segment, segments */
void emu_plan_wbfm(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count, uint32_t *out4)
{
    const b200::FmPlan pl = b200::plan_wbfm_batch(len_bytes, n_captures, sm_count);
    out4[0] = pl.n_tiles;
    out4[1] = pl.total_chunks;
    out4[2] = pl.tiles_per_segment;
    out4[3] = pl.segments;
}

/* the tensor-core WBFM plan: out5 = n_tiles, total_rows, tiles_per_segment, segments, grid */
void emu_plan_wbfm_tc(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count, uint32_t *out5)
{
    const b200::FmTcPlan pl = b200::plan_wbfm_tc(len_bytes, n_captures, sm_count);
    out5[0] = pl.n_tiles;
    out5[1] = pl.total_rows;
    out5[2] = pl.tiles_per_segment;
    out5[3] = pl.segments;
    out5[4] = pl.grid;
}

/* the AM batch plan: out5 = n_tiles, total_chunks, tiles_per_segment, segments, q_count */
void emu_plan_am(uint64_t len_bytes, uint32_t n_captures, uint32_t sm_count, uint32_t *out5)
{
    const b200::AmPlan pl = b200::plan_am_batch(len_bytes, n_captures, sm_count);
    out5[0] = pl.n_tiles;
    out5[1] = pl.total_chunks;
    out5[2] = pl.tiles_per_segment;
    out5[3] = pl.segments;
    out5[4] = (uint32_t)pl.q_count;
}

} /* extern "C" */
