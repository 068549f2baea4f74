/* Test harness (plain C, not part of libb200g16): the declarations of the group batch prove (b200g16_bases_copy,
 * b200g16_group_pk_replicate, b200g16_group_prove_batch) compile as C11, link, and refuse NULL arguments without
 * touching a device.  Built and run by tests/test_group_batch_cpu.py. */
#include <stdio.h>
#include <string.h>

#include "b200g16.h"

int main(void) {
  b200g16_bases* bout = NULL;
  b200g16_group_pk* gout = NULL;
  b200g16_proof proof;
  uint64_t word[4] = {0, 0, 0, 0};
  memset(&proof, 0, sizeof proof);
  if (b200g16_bases_copy(NULL, NULL, &bout) != B200G16_ERR_ARG || bout) return 10;
  if (b200g16_bases_copy(NULL, NULL, NULL) != B200G16_ERR_ARG) return 11;
  if (b200g16_group_pk_replicate(NULL, NULL, &gout) != B200G16_ERR_ARG || gout) return 12;
  if (b200g16_group_prove_batch(NULL, NULL, 0, NULL, 0, NULL, NULL, NULL, 0, NULL, NULL, NULL) != B200G16_ERR_ARG)
    return 13;
  if (b200g16_group_prove_batch(NULL, NULL, 1, word, 1, word, word, word, 1, word, word, &proof) != B200G16_ERR_ARG)
    return 14;
  if (strlen(b200g16_last_error()) == 0) return 15;
  b200g16_group_pk_free(NULL);
  printf("ok: %s\n", b200g16_last_error());
  return 0;
}
