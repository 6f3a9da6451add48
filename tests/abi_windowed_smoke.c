/* tests/abi_windowed_smoke.c -- windowed MSM bases (d377_msm_bases_create_windowed) driven
 * from a plain C host: create a set, run MSMs over it through the blocking and the pipelined
 * entry points, read its layout, destroy it twice.  Compiled with gcc and linked against
 * decaf377_b200/libdecaf377_b200.so by tests/test_gpu_windowed_bases.py.  The points are
 * i*G, i = 0..15, decompressed from the encodings the reference's tests hold
 * (tests/encoding.rs:61-78); results are checked against those encodings and against the
 * MSM over the same Elements without prepared bases. */
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "decaf377_b200.h"

static int failures = 0;
#define CHECK(cond)                                                              \
  do {                                                                           \
    if (!(cond)) {                                                               \
      printf("FAIL %s:%d: %s  [%s]\n", __FILE__, __LINE__, #cond, d377_last_error()); \
      failures++;                                                                \
    }                                                                            \
  } while (0)
#define OK(call) CHECK((call) == D377_OK)

/* encodings of 0, G, 3G, 15G (tests/encoding.rs) */
static const uint8_t ENC0[32] = {0};
static const uint8_t ENC1[32] = {0x08};
static const uint8_t ENC3[32] = {0x2e, 0xbd, 0x42, 0xdd, 0x3a, 0x23, 0x07, 0x08, 0x3c, 0x83, 0x4e, 0x79, 0xfb, 0x9e, 0x78, 0x7e,
                                 0x35, 0x2d, 0xd3, 0x3e, 0x0d, 0x71, 0x9f, 0x86, 0xae, 0x4a, 0xdb, 0x02, 0xfe, 0x38, 0x24, 0x09};
static const uint8_t ENC15[32] = {0xbc, 0xb0, 0xf9, 0x22, 0xdf, 0x1c, 0x7a, 0xa9, 0x57, 0x93, 0x94, 0x02, 0x01, 0x87, 0xa2, 0xe1,
                                  0x9e, 0x2d, 0x80, 0x73, 0x45, 0x2c, 0x6a, 0xb9, 0xb0, 0xc4, 0xb0, 0x52, 0xaa, 0x50, 0xf5, 0x05};

enum { N = 16 };

int main(void) {
  OK(d377_init(0));
  /* points i*G: 0 -> identity, 1 -> G, 3 -> 3G, 15 -> 15G; the rest are multiples of G too,
   * produced by the library (fixed-base multiplication) */
  uint8_t sc1[N * 32], enc[N * 32], el[N * 128], ok[N];
  memset(sc1, 0, sizeof sc1);
  for (int i = 0; i < N; i++) sc1[32 * i] = (uint8_t)i;
  OK(d377_fixed_base_mul(sc1, N, enc, 1));
  CHECK(memcmp(enc, ENC0, 32) == 0 && memcmp(enc + 32, ENC1, 32) == 0);
  CHECK(memcmp(enc + 96, ENC3, 32) == 0 && memcmp(enc + 32 * 15, ENC15, 32) == 0);
  OK(d377_batch_decompress(enc, N, el, ok));
  /* scalars: s_3 = 5, all others 0 -> 15G */
  uint8_t sc[N * 32], got[32], want[32];
  memset(sc, 0, sizeof sc);
  sc[32 * 3] = 5;
  uint8_t* win = NULL;
  OK(d377_msm_bases_create_windowed(el, D377_PT_ELEMENT, N, 7, &win));
  OK(d377_msm(sc, win, D377_PT_BASES, N, NULL, got));
  CHECK(memcmp(got, ENC15, 32) == 0);
  /* dense scalars with digits in every window: same result as the plain MSM */
  for (int i = 0; i < N * 32; i++) sc[i] = (uint8_t)(37 * i + 11);
  for (int i = 0; i < N; i++) sc[32 * i + 31] = 0x03;   /* < r */
  OK(d377_msm(sc, el, D377_PT_ELEMENT, N, NULL, want));
  OK(d377_msm(sc, win, D377_PT_BASES, N, NULL, got));
  CHECK(memcmp(got, want, 32) == 0);
  /* pipelined form, a prefix, and a pointer into the middle of the set */
  OK(d377_msm_submit(sc, win, D377_PT_BASES, N, 0));
  OK(d377_msm_wait(0, NULL, got));
  CHECK(memcmp(got, want, 32) == 0);
  OK(d377_msm(sc, el, D377_PT_ELEMENT, 5, NULL, want));
  OK(d377_msm(sc, win, D377_PT_BASES, 5, NULL, got));
  CHECK(memcmp(got, want, 32) == 0);
  CHECK(d377_msm(sc, win + 128, D377_PT_BASES, 4, NULL, got) == D377_ERR_INVALID_ARG);
  CHECK(d377_msm(sc, win, D377_PT_BASES, N + 1, NULL, got) == D377_ERR_INVALID_ARG);
  /* layout */
  size_t n = 0, bytes = 0;
  int c = 0, w = 0;
  OK(d377_msm_bases_info(win, &n, &c, &w, &bytes));
  CHECK(n == N && c == 7 && w == 36 && bytes >= (size_t)N * 36 * 128);
  /* argument checks */
  uint8_t* bad = NULL;
  CHECK(d377_msm_bases_create_windowed(el, D377_PT_ELEMENT, N, 3, &bad) == D377_ERR_INVALID_ARG);
  CHECK(d377_msm_bases_create_windowed(el, D377_PT_ELEMENT, N, 23, &bad) == D377_ERR_INVALID_ARG);
  CHECK(bad == NULL);
  OK(d377_msm_bases_destroy(win));
  CHECK(d377_msm_bases_destroy(win) == D377_ERR_INVALID_ARG);
  CHECK(d377_msm_bases_info(win, &n, &c, &w, &bytes) == D377_ERR_INVALID_ARG);
  OK(d377_shutdown());
  if (failures) {
    printf("abi_windowed_smoke: %d check(s) failed\n", failures);
    return 1;
  }
  printf("abi_windowed_smoke: all checks passed\n");
  return 0;
}
