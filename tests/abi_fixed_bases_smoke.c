/* tests/abi_fixed_bases_smoke.c -- prepared fixed bases (d377_fixed_bases_create) driven from a
 * plain C host: create a set of k = 2 bases from their encodings, run linear combinations
 * through the host and device entry points, read the set's layout, check the refusals, destroy
 * it twice.  Compiled with gcc -Wall -Werror and linked against
 * decaf377_b200/libdecaf377_b200.so by tests/test_gpu_fixed_bases.py (and, without a GPU, by
 * tests/test_fixed_bases_cpu.py, where it must fail loudly).  The bases are G and 3G, given by
 * the encodings the reference's tests hold (tests/encoding.rs:61-78); results are checked
 * against those encodings and against d377_fixed_base_mul. */
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

enum { N = 4, K = 2 };

int main(void) {
  OK(d377_init(0));
  uint8_t bases_enc[K * 32];
  memcpy(bases_enc, ENC1, 32);
  memcpy(bases_enc + 32, ENC3, 32);
  uint8_t* fb = NULL;
  OK(d377_fixed_bases_create(bases_enc, D377_PT_ENCODING, K, &fb));
  CHECK(fb != NULL);
  size_t k = 0, bytes = 0;
  OK(d377_fixed_bases_info(fb, &k, &bytes));
  CHECK(k == K && bytes == (size_t)K * (16 * 32768 + 1) * 96);
  /* rows (a, b) -> a G + b 3G: (0, 0) -> 0, (1, 0) -> G, (0, 5) -> 15G, (12, 1) -> 15G */
  uint8_t sc[N * K * 32], enc[N * 32];
  memset(sc, 0, sizeof sc);
  sc[(1 * K + 0) * 32] = 1;
  sc[(2 * K + 1) * 32] = 5;
  sc[(3 * K + 0) * 32] = 12;
  sc[(3 * K + 1) * 32] = 1;
  OK(d377_fixed_bases_mul(fb, sc, N, enc, D377_OUT_ENCODING));
  CHECK(memcmp(enc, ENC0, 32) == 0 && memcmp(enc + 32, ENC1, 32) == 0);
  CHECK(memcmp(enc + 64, ENC15, 32) == 0 && memcmp(enc + 96, ENC15, 32) == 0);
  /* Element output, compressed, gives the same bytes */
  uint8_t el[N * 128], enc2[N * 32];
  OK(d377_fixed_bases_mul(fb, sc, N, el, D377_OUT_ELEMENT));
  OK(d377_batch_compress(el, N, enc2));
  CHECK(memcmp(enc, enc2, sizeof enc) == 0);
  /* k = 1 over G itself equals the generator path */
  uint8_t* g = NULL;
  OK(d377_fixed_bases_create(ENC1, D377_PT_ENCODING, 1, &g));
  uint8_t s1[32 * 3], want[32 * 3], got[32 * 3];
  for (int i = 0; i < (int)sizeof s1; i++) s1[i] = (uint8_t)(29 * i + 3);
  OK(d377_fixed_base_mul(s1, 3, want, D377_OUT_ENCODING));
  OK(d377_fixed_bases_mul(g, s1, 3, got, D377_OUT_ENCODING));
  CHECK(memcmp(got, want, sizeof got) == 0);
  /* n = 0 is a no-op */
  OK(d377_fixed_bases_mul(fb, sc, 0, enc, D377_OUT_ENCODING));
  /* refusals: k = 0, bad formats, null pointers, foreign handles */
  uint8_t* bad = NULL;
  CHECK(d377_fixed_bases_create(bases_enc, D377_PT_ENCODING, 0, &bad) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_create(bases_enc, D377_PT_BASES, K, &bad) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_create(NULL, D377_PT_ENCODING, K, &bad) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_create(bases_enc, D377_PT_ENCODING, K, NULL) == D377_ERR_INVALID_ARG);
  uint8_t invalid[32] = {1};   /* tests/encoding.rs:28-52 */
  CHECK(d377_fixed_bases_create(invalid, D377_PT_ENCODING, 1, &bad) == D377_ERR_INVALID_ENCODING);
  CHECK(bad == NULL);
  CHECK(d377_fixed_bases_mul(fb, sc, N, enc, 2) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_mul(fb, NULL, N, enc, D377_OUT_ENCODING) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_mul(fb + 96, sc, N, enc, D377_OUT_ENCODING) == D377_ERR_INVALID_ARG);
  uint8_t* msm = NULL;
  OK(d377_msm_bases_create(bases_enc, D377_PT_ENCODING, K, &msm));
  CHECK(d377_fixed_bases_mul(msm, sc, N, enc, D377_OUT_ENCODING) == D377_ERR_INVALID_ARG);
  CHECK(d377_msm(sc, fb, D377_PT_BASES, K, NULL, enc) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_destroy(msm) == D377_ERR_INVALID_ARG);
  OK(d377_msm_bases_destroy(msm));
  OK(d377_fixed_bases_destroy(fb));
  CHECK(d377_fixed_bases_destroy(fb) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_info(fb, &k, &bytes) == D377_ERR_INVALID_ARG);
  CHECK(d377_fixed_bases_mul(fb, sc, N, enc, D377_OUT_ENCODING) == D377_ERR_INVALID_ARG);
  /* shutdown releases the set still alive */
  OK(d377_shutdown());
  if (failures) {
    printf("abi_fixed_bases_smoke: %d check(s) failed\n", failures);
    return 1;
  }
  printf("abi_fixed_bases_smoke: all checks passed\n");
  return 0;
}
