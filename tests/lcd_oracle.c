/* lcd_oracle.c -- CPU restatement of the loop-closure candidates and word weights (include/maveric_b200.h,
 * mv_loop_candidates and mv_lcd_word_weights; DESIGN §4.7).  TEST INFRASTRUCTURE ONLY, built by tests/lcd_oracle.py.
 *
 * Plain loops, written apart from the GPU's GEMM formulation: every frame's valid words are reduced to a sorted list
 * of distinct ids (the form lcd_main.c intersects), a posting list per word gives the frames that hold it, and the
 * score of (i, j) is accumulated word by word over i's list.  The top k is a repeated arg-max with the smaller j on
 * equal scores. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int cmp_int(const void* a, const void* b) {
  const int x = *(const int*)a, y = *(const int*)b;
  return (x > y) - (x < y);
}

/* distinct valid words of every frame, sorted: list[f] = ids[off[f] .. off[f + 1]) */
static void distinct_words(int n, int top_n, int n_words, const int32_t* word, const int32_t* q_count, int** ids_out,
                           long long** off_out) {
  long long* off = (long long*)malloc(sizeof(long long) * (size_t)(n + 1));
  int* ids = (int*)malloc(sizeof(int) * ((size_t)n * top_n + 1));
  off[0] = 0;
  for (int f = 0; f < n; f++) {
    int nq = q_count[f] < 0 ? 0 : q_count[f];
    if (nq > top_n) nq = top_n;
    int* l = ids + off[f];
    int m = 0;
    for (int q = 0; q < nq; q++) {
      const int w = word[(size_t)f * top_n + q];
      if (w >= 0 && w < n_words) l[m++] = w;
    }
    qsort(l, (size_t)m, sizeof(int), cmp_int);
    int d = 0;
    for (int q = 0; q < m; q++)
      if (d == 0 || l[d - 1] != l[q]) l[d++] = l[q];
    off[f + 1] = off[f] + d;
  }
  *ids_out = ids;
  *off_out = off;
}

void orc_lcd_candidates(int n, int first_frame, int top_n, int n_words, const int32_t* word, const int32_t* q_count,
                        const int8_t* weight /* nullable: all 1 */, int min_gap, int k, int min_score, int32_t* cand,
                        int32_t* score) {
  int* ids;
  long long* off;
  distinct_words(n, top_n, n_words, word, q_count, &ids, &off);
  /* posting lists: the frames holding each word, ascending */
  long long* pstart = (long long*)calloc((size_t)n_words + 1, sizeof(long long));
  for (long long e = 0; e < off[n]; e++) pstart[ids[e] + 1]++;
  for (int w = 0; w < n_words; w++) pstart[w + 1] += pstart[w];
  long long* fill = (long long*)malloc(sizeof(long long) * (size_t)n_words);
  memcpy(fill, pstart, sizeof(long long) * (size_t)n_words);
  int* post = (int*)malloc(sizeof(int) * ((size_t)off[n] + 1));
  for (int f = 0; f < n; f++)
    for (long long e = off[f]; e < off[f + 1]; e++) post[fill[ids[e]]++] = f;

  int* s = (int*)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  unsigned char* taken = (unsigned char*)malloc((size_t)(n > 0 ? n : 1));
  for (int i = 0; i < n; i++) {
    const long long hi = (long long)i - min_gap;   /* allowed j: 0 .. hi */
    for (int r = 0; r < k; r++) {
      cand[(size_t)i * k + r] = -1;
      score[(size_t)i * k + r] = 0;
    }
    if (hi < 0) continue;
    for (long long j = 0; j <= hi; j++) { s[j] = 0; taken[j] = 0; }
    for (long long e = off[i]; e < off[i + 1]; e++) {
      const int w = ids[e];
      const int wt = weight ? weight[w] : 1;
      for (long long p = pstart[w]; p < pstart[w + 1] && post[p] <= hi; p++) s[post[p]] += wt;
    }
    for (int r = 0; r < k; r++) {
      long long best = -1;
      for (long long j = 0; j <= hi; j++)
        if (!taken[j] && s[j] >= min_score && (best < 0 || s[j] > s[best])) best = j;
      if (best < 0) break;
      taken[best] = 1;
      cand[(size_t)i * k + r] = first_frame + (int)best;
      score[(size_t)i * k + r] = s[best];
    }
  }
  free(s); free(taken); free(post); free(fill); free(pstart); free(ids); free(off);
}

void orc_lcd_word_weights(int n, int top_n, int n_words, const int32_t* word, const int32_t* q_count, int8_t* weight) {
  int* ids;
  long long* off;
  distinct_words(n, top_n, n_words, word, q_count, &ids, &off);
  int* df = (int*)calloc((size_t)n_words, sizeof(int));
  for (long long e = 0; e < off[n]; e++) df[ids[e]]++;
  for (int w = 0; w < n_words; w++)
    weight[w] = df[w] ? (int8_t)rint(127.0 * log((double)n / (double)df[w]) / log((double)n)) : (int8_t)0;
  free(df); free(ids); free(off);
}
