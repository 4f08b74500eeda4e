/* ctxnerf_diag.h -- diagnostics build of the library (libctxnerf_diag.so = the product sources compiled with
 * -DCTXNERF_DIAG + csrc/diag/tc_selftest.cu).  None of this is part of the drop-in boundary (include/ctxnerf.h):
 * tcgen05 / mbarrier micro-benchmarks, one-CTA GEMM self-tests that pin the descriptor conventions, the hooks of
 * the profiling instantiation of the forward kernel (per-role cycle counters, deadlock reporter) and the dgrad
 * kernel's per-role cycle counters.  Used by tools/ and by one GPU test; the product library exports none of these
 * symbols.                                                                                                      */
#ifndef CTXNERF_DIAG_H
#define CTXNERF_DIAG_H
#include "ctxnerf.h"
#ifdef __cplusplus
extern "C" {
#endif

/* profiling instantiation of ctx_mlp_fwd: 16 x uint64 cycle counters per CTA (device pointer; NULL = off) */
int ctx_mlp_set_prof_buffer(void* device_u64);
/* 1 = epilogue skips the TMEM loads / stores, 2 = issuer skips the MMAs (timing experiments) */
int ctx_mlp_set_debug(int flags);
/* pinned host buffer the kernel's waiters report into before trapping when a barrier wait exceeds ~0.2 s */
int ctx_mlp_set_hang_buffer(void* pinned_u64);
/* dgrad kernel: 16 x uint64 per-role cycle counters per CTA (device pointer; NULL = off) */
int ctx_dgrad_set_prof(void* device_u64);

/* diagnostic: one-CTA tcgen05 GEMM C[128,N] = A * B^T (tests pin the descriptor
 * conventions with it); A,B bf16.  mode 0 K-major operands, 1 MN-major.          */
int ctx_tcgen05_selftest(const void* A, const void* B, float* C, int N, int K, int mode, int variant,
                         void* stream);
/* same through a 2-CTA cluster: C[256,N] with tcgen05.mma.cta_group::2 (M = 256) */
int ctx_tcgen05_selftest2(const void* A, const void* B, float* C, int N, int K, void* stream);

/* back-to-back tcgen05.mma rate / mbarrier + fence issue costs (profiles/microbench_r01.md) */
int ctx_tcgen05_mma_rate(int two_cta, int n_mma, int N, int n_ctas, void* out_cycles, int mode, const void* src,
                         void* stream);
int ctx_tcgen05_sync_cost(void* out_cycles, int reps, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTXNERF_DIAG_H */
