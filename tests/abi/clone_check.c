/* clone_check.c -- plain C99 against include/blu_b200.h: factorizes the 10 x 10 example of abi_check.c, clones the
 * object, saves it to an image and restores that into a third object, and checks that all three give the same solution
 * bit for bit and that a clone of a batch is refused.
 * Build: gcc -std=c99 -I include tests/abi/clone_check.c -L <dir> -l<library> -Wl,-rpath,<dir> */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "blu_b200.h"

int main(void) {
    static const int64_t bp[11] = {0, 3, 6, 8, 13, 15, 16, 19, 23, 27, 32};
    static const int64_t bi[32] = {0, 7, 8, 1, 4, 9, 2, 9, 3, 6, 7, 8, 9, 1, 4, 5, 3, 6, 9, 0, 3, 7, 8, 0, 3, 7, 8, 1, 2, 3, 6, 9};
    static const double bx[32] = {2.1, 0.14, 0.09, 1.1, 0.06, 0.03, 1.7, 0.04, 1.0, 0.32, 0.19, 0.32, 0.44, 0.06, 1.6, 2.2, 0.32, 1.9, 0.43,
                                  0.14, 0.19, 1.1, 0.22, 0.09, 0.32, 0.22, 2.4, 0.03, 0.04, 0.44, 0.43, 3.2};
    double rhs[10], x0[10], x1[10], x2[10];
    blu_t *o = NULL, *c = NULL, *r = NULL;
    blu_batch_t *b = NULL;
    int64_t bytes = 0;
    unsigned char *raw;
    void *img;
    int k;
    if (blu_create(&o, 10, 32, -1) != BLU_OK || blu_factorize(o, bp, bp + 1, bi, bx) != BLU_OK) { printf("set-up failed\n"); return 1; }
    for (k = 0; k < 10; k++) rhs[k] = 1.0 + 0.5 * (double)k;
    if (blu_clone(&c, o) != BLU_OK) { printf("blu_clone failed\n"); return 1; }
    if (blu_save(o, NULL, 0, &bytes) != BLU_OK || bytes <= 0) { printf("blu_save size query failed\n"); return 1; }
    raw = malloc((size_t)bytes + 16);
    if (!raw) return 1;
    img = raw + (16 - (size_t)raw % 16) % 16;      /* 16-byte aligned */
    if (blu_save(o, img, bytes, &bytes) != BLU_OK) { printf("blu_save failed\n"); return 1; }
    if (blu_create(&r, 10, 4, -1) != BLU_OK || blu_restore(r, img, bytes) != BLU_OK) { printf("blu_restore failed\n"); return 1; }
    if (blu_solve_dense(o, rhs, x0, 'N') != BLU_OK || blu_solve_dense(c, rhs, x1, 'N') != BLU_OK || blu_solve_dense(r, rhs, x2, 'N') != BLU_OK) {
        printf("solve failed\n");
        return 1;
    }
    if (memcmp(x0, x1, sizeof x0) || memcmp(x0, x2, sizeof x0)) { printf("solutions differ\n"); return 1; }
    if (blu_batch_create(&b, 2, 10, 32, -1) != BLU_OK) { printf("blu_batch_create failed\n"); return 1; }
    if (blu_clone(&c, b) != BLU_ERROR_INVALID_ARGUMENT) { printf("a batch was cloned\n"); return 1; }
    printf("clone and image of the 10 x 10 example solve alike (%lld image bytes)\n", (long long)bytes);
    blu_batch_destroy(b);
    blu_destroy(r);
    blu_destroy(c);
    blu_destroy(o);
    free(raw);
    return 0;
}
