/* hypernerf_b200_probe — microbenchmark / descriptor-probe / profiling entry points.
 *
 * NOT part of the drop-in boundary (include/hypernerf_b200.h): nothing here replaces a reference function.  These are
 * built into their own shared object, libhypernerf_b200_probe.so, used by tests/test_probe.py (pins the UMMA shared-memory
 * descriptor conventions of hn_ptx.cuh against a plain matmul) and by the measurement scripts under profiles/.
 * hn_debug_set_timing_buffer is exported by the role-timing builds of the main library only (make timing /
 * -DHN_ROLE_TIMING=1, selected at run time with HN_LIB). */
#ifndef HYPERNERF_B200_PROBE_H
#define HYPERNERF_B200_PROBE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* test hook: one UMMA tile D[128,N] = A * B^T through the shared-memory layouts the MLP kernels use.
 * a_mn / b_mn = 0: operand given row-major [rows][K]; 1: given as [K][rows] (MN-major). */
int hn_umma_probe(const void* A_bf16, const void* B_bf16, float* D, int N, int K, int a_mn, int b_mn, void* stream);

/* test hook: D[256,N] = A[256,K] * B[N,K]^T on a 2-CTA cluster with cta_group::2 (A, B row-major [rows][K]). */
int hn_umma_probe2(const void* A_bf16, const void* B_bf16, float* D, int N, int K, void* stream);

/* test hook: cycles for reps x (inner x ksteps x nsub back-to-back K=16 UMMAs (M=128) + one commit/wait) from resident
 * shared-memory operands; swizzle 0 = un-swizzled interleave layout, 1 = 128B swizzle.  out_cycles: uint64 per CTA. */
int hn_umma_rate(int N, int ksteps, int reps, int swizzle, int nsub, int inner, int grid, void* out_cycles, void* stream);

/* test hook: per-UMMA cost by accumulator rotation (nacc, order), M, A source (0 smem, 1 same smem slice, 2 TMEM) and
 * CTA pairing (cta_group 1, or 2 on a 2-CTA cluster); reps x (inner x 16 x nacc UMMAs + commit/wait). */
int hn_umma_rate2(int cta_group, int M, int N, int nacc, int order, int a_src, int reps, int inner, int grid,
                  void* out_cycles, void* stream);

/* test hook: as hn_umma_rate but a fully unrolled issue sequence (N in {16,64,128,256}, nacc in {1,2}). */
int hn_umma_rate3(int N, int nacc, int reps, int inner, int grid, void* out_cycles, void* stream);

/* test hook: cycles for 8 warps to drain a 256-column accumulator with a selectable subset of the epilogue's work. */
int hn_epi_rate(int mode, int reps, int grid, void* gout, void* out_cycles, void* stream);

/* test hook: as hn_umma_rate3 for the CTA-pair form (cta_group::2, M = 256 on 2-CTA clusters). */
int hn_umma_rate4(int N, int nacc, int reps, int inner, int grid, void* out_cycles, void* stream);

/* test hook: cycles for nwarps warps to read `cols` TMEM columns of their 32 lanes `reps` times (tcgen05.ld.32x32b.x32). */
int hn_tmem_rate(int nwarps, int cols, int reps, int mode, void* out_cycles, void* stream);

/* test hook: four warps drain a 128 x 256 accumulator `reps` times (mode bits: 1 bf16 pack, 2 st.shared, 4 st.global, 8 bias)
 * while (umma != 0) another warp issues back-to-back M = 128, N = umma_n UMMAs and (tma != 0) a third keeps re-loading a
 * 16 KB stage by bulk copies.  gout: grid x 64 KB, gsrc: 1 MB, out: 4 x uint64 per CTA {drain cycles, UMMAs retired,
 * issuer cycles, bulk copies}. */
int hn_overlap_rate(int mode, int umma, int umma_n, int tma, int reps, int grid, void* gout, const void* gsrc, void* out,
                    void* stream);

/* profiling hook: device buffer of 8 x uint64 per CTA filled by the fused MLP kernels with per-role cycle counters
 * (producer wait, UMMA-issuer waits, epilogue wait / work); NULL = off. */
int hn_debug_set_timing_buffer(void* dev_buffer);

#ifdef __cplusplus
}
#endif
#endif /* HYPERNERF_B200_PROBE_H */
