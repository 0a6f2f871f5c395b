/*
 * sslam_b200_debug.h — debug aids exported by libsslam_b200.so for the probes under tools/.
 * NOT part of the drop-in ABI (include/sslam_b200.h); signatures may change without an ABI bump.
 */
#ifndef SSLAM_B200_DEBUG_H_
#define SSLAM_B200_DEBUG_H_

#ifdef __cplusplus
extern "C" {
#endif

/* Host-mapped buffer (device pointer) that receives {block, thread, barrier, parity} records of
 * mbarrier waits that timed out in the GEMM translation unit; returns a cudaError_t value. */
int sslam_debug_watchdog_gemm(unsigned long long* buf);

/* 0: force the register-prefetching decode scan + radix-select top-k (the fallback kernels for maps the
 * streaming scan does not take); non-zero (default): streaming scan + histogram top-k where eligible. */
void sslam_debug_decode_stream(int on);

/* Streaming decode scan: stages of the shared-memory ring per CTA and rows per band (0 = library default). */
void sslam_debug_decode_tune(int stages, int band_rows);

/* DescriptorRefiner forward: 0 = one GEMM launch per layer; 1..4 = the layer-fused persistent kernel with
 * that many 256-row strip pairs per chunk (default 3).  Other values are clamped to 0..4.  Both paths
 * compute bit-identical results. */
void sslam_debug_refiner_fused(int mode);

#ifdef __cplusplus
}
#endif
#endif /* SSLAM_B200_DEBUG_H_ */
