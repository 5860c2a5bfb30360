/*
 * topk_ref.c — CPU reference of gdr_topk_scores for the tests.  Plain sequential arithmetic:
 *   s(u, j) = acc = 0; for t < d: acc = fmaf(U[u, t], I[j, t], acc)
 * glibc's fmaf rounds correctly, so every score is bit-equal to CUDA's fmaf chain.  Items are ordered by
 * (score desc, item asc) with a comparison sort (-0 reported as +0); excluded items never appear; rows with
 * fewer than k eligible items are padded with (-1, -inf).  OpenMP splits rows only.
 *
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC topk_ref.c -o libtopk_ref.so -lm
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

typedef struct {
  float s;
  int32_t j;
} pair_t;

static int cmp_pair(const void* a, const void* b) {
  const pair_t* x = (const pair_t*)a;
  const pair_t* y = (const pair_t*)b;
  if (x->s > y->s) return -1;
  if (x->s < y->s) return 1;
  return (x->j > y->j) - (x->j < y->j);
}

void ref_topk(int64_t n_rows, int64_t n_items, int64_t d, int64_t k, const float* U, int64_t ldu,
              const int64_t* rows, const float* I, int64_t ldi, const int32_t* ex_rowptr, const int32_t* ex_colidx,
              float* scores_out, int32_t* items_out) {
#pragma omp parallel
  {
    pair_t* p = (pair_t*)malloc(sizeof(pair_t) * (size_t)n_items);
    char* excl = (char*)malloc((size_t)n_items);
#pragma omp for schedule(dynamic, 4)
    for (int64_t r = 0; r < n_rows; ++r) {
      const int64_t u = rows ? rows[r] : r;
      for (int64_t j = 0; j < n_items; ++j) excl[j] = 0;
      if (ex_rowptr)
        for (int32_t e = ex_rowptr[u]; e < ex_rowptr[u + 1]; ++e) excl[ex_colidx[e]] = 1;
      int64_t m = 0;
      for (int64_t j = 0; j < n_items; ++j) {
        if (excl[j]) continue;
        float acc = 0.0f;
        for (int64_t t = 0; t < d; ++t) acc = fmaf(U[u * ldu + t], I[j * ldi + t], acc);
        p[m].s = acc + 0.0f;
        p[m].j = (int32_t)j;
        ++m;
      }
      qsort(p, (size_t)m, sizeof(pair_t), cmp_pair);
      for (int64_t i = 0; i < k; ++i) {
        scores_out[r * k + i] = i < m ? p[i].s : -INFINITY;
        items_out[r * k + i] = i < m ? p[i].j : -1;
      }
    }
    free(p);
    free(excl);
  }
}
