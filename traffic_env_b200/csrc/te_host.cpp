// te_host.cpp - host side of the wire format (te_kernels.cuh: wire_layout): expand compact env records
//   u8 passed[r] | u8 detected[r] | f32 light[I] | f32 reward[I] | u8 done
// into the float observation / reward / done arrays te_step returns (traffic_test.py:37-56: Repeater's total_obs is
// float32[2r + I]).  Memory-bound; an AVX2 path with streaming stores is picked at run time when the CPU has it.
#include <cstdint>
#include <cstring>
#include <immintrin.h>

#include "../../include/traffic_b200.h"

namespace {

void expand_scalar(const unsigned char *__restrict__ rec, int n, float *__restrict__ out) {
  for (int k = 0; k < n; k++) out[k] = (float)rec[k];
}

// Long rows (10x10 grid: 800 counts per env): streaming stores - the expanded observation is written once and read
// later by somebody else, so it should not displace the reader's working set nor cost a read-for-ownership.
__attribute__((target("avx2"))) void expand_avx2_stream(const unsigned char *__restrict__ rec, int n, float *__restrict__ out) {
  int k = 0;
  // head: up to the first 32-byte boundary of the destination
  while (k < n && (reinterpret_cast<uintptr_t>(out + k) & 31u)) { out[k] = (float)rec[k]; k++; }
  for (; k + 8 <= n; k += 8) {
    const __m128i b = _mm_loadl_epi64(reinterpret_cast<const __m128i *>(rec + k));
    _mm256_stream_ps(out + k, _mm256_cvtepi32_ps(_mm256_cvtepu8_epi32(b)));
  }
  for (; k < n; k++) out[k] = (float)rec[k];
}

// Short rows (default grid: 72 counts per env, the float light term follows in the same cache lines): plain
// unaligned stores - streaming stores that share cache lines with ordinary ones are slow.
__attribute__((target("avx2"))) void expand_avx2(const unsigned char *__restrict__ rec, int n, float *__restrict__ out) {
  int k = 0;
  for (; k + 8 <= n; k += 8) {
    const __m128i b = _mm_loadl_epi64(reinterpret_cast<const __m128i *>(rec + k));
    _mm256_storeu_ps(out + k, _mm256_cvtepi32_ps(_mm256_cvtepu8_epi32(b)));
  }
  for (; k < n; k++) out[k] = (float)rec[k];
}

bool have_avx2() {
  static const bool v = __builtin_cpu_supports("avx2");
  return v;
}

}  // namespace

void te_expand_records_host(const unsigned char *recs, const te_wire_layout_t &wl, int r, int I, long long n, float *obs,
                            float *reward, uint8_t *done) {
  const int ol = 2 * r + I;
  const bool avx2 = have_avx2();
  const bool stream = avx2 && 2 * r >= 512;
  for (long long e = 0; e < n; e++) {
    const unsigned char *rec = recs + (size_t)e * wl.stride;
    float *o = obs + (size_t)e * ol;
    // passed and detected: one run of 2r counts (detected follows passed in the record as in the observation)
    if (stream) expand_avx2_stream(rec + wl.passed, 2 * r, o);
    else if (avx2) expand_avx2(rec + wl.passed, 2 * r, o);
    else expand_scalar(rec + wl.passed, 2 * r, o);
    // light term and reward: I floats each (4-byte aligned inside the record)
    const float *__restrict__ lf = reinterpret_cast<const float *>(rec + wl.light);
    const float *__restrict__ rf = reinterpret_cast<const float *>(rec + wl.reward);
    float *__restrict__ ol_ = o + 2 * r;
    float *__restrict__ rw = reward + (size_t)e * I;
    if (I <= 32) {            // small grids: a library memcpy call per 36 bytes costs more than the copy
      for (int i = 0; i < I; i++) ol_[i] = lf[i];
      for (int i = 0; i < I; i++) rw[i] = rf[i];
    } else {
      memcpy(ol_, lf, (size_t)I * 4);
      memcpy(rw, rf, (size_t)I * 4);
    }
    done[e] = rec[wl.done];
  }
  if (stream) _mm_sfence();
}
