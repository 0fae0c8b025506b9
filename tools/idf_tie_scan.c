/* idf_tie_scan.c -- how close the idf weight of mv_lcd_word_weights comes to a rounding tie, over every (n, df)
 * with 2 <= n <= 65 535 and 1 <= df <= n.
 *
 *   gcc -std=gnu11 -O2 -fopenmp -ffp-contract=off -o /tmp/idf_tie_scan tools/idf_tie_scan.c -lm && /tmp/idf_tie_scan
 *
 * The weight is rint(127 ln(n / df) / ln(n)) evaluated in double.  Its exact value is a half-integer only at
 * df^2 = n (63.5; the proof is beside word_weights_kernel in csrc/lcd.cu), which the library decides in integers.
 * This prints, with the C library's log: at each of those ties, what the double evaluation gives; and over every
 * other (n, df) the least distance of the double value from a half-integer, for n up to 4 541 (the bench sequence's
 * length) and up to 65 535 (the limit).  A distance many ulp wide means an evaluation whose log is off by an ulp or
 * two (the device's) rounds every such value the same way as the host's. */
#include <math.h>
#include <stdio.h>

#define N_MAX 65535

int main(void) {
  int off = 0, low = 0;
  for (int m = 2; m * m <= N_MAX; m++) {
    const int n = m * m;
    const double v = 127.0 * log((double)n / (double)m) / log((double)n);
    if (v != 63.5) off++;
    if (rint(v) != 64.0) low++;
  }
  printf("ties df^2 = n, m = 2 .. 255: the double value is not 63.5 at %d of 254, and rint gives 63 at %d\n", off, low);

  static double best[N_MAX + 1];
  static int best_df[N_MAX + 1];
#pragma omp parallel for schedule(dynamic, 64)
  for (int n = 2; n <= N_MAX; n++) {
    const double ln = log((double)n);
    double b = 1.0;
    int bd = 0;
    for (int df = 1; df <= n; df++) {
      if ((long long)df * df == n) continue;
      const double v = 127.0 * log((double)n / (double)df) / ln;
      const double d = fabs(v - floor(v) - 0.5);
      if (d < b) { b = d; bd = df; }
    }
    best[n] = b;
    best_df[n] = bd;
  }
  const int limits[2] = {4541, N_MAX};
  for (int l = 0; l < 2; l++) {
    int bn = 2;
    for (int n = 2; n <= limits[l]; n++)
      if (best[n] < best[bn]) bn = n;
    const double v = 127.0 * log((double)bn / (double)best_df[bn]) / log((double)bn);
    printf("n <= %d, df^2 != n: least distance from a half-integer %.3e at n = %d, df = %d (value %.17g; %.0f ulp "
           "of 64)\n", limits[l], best[bn], bn, best_df[bn], v, best[bn] / ldexp(1.0, -46));
  }
  return 0;
}
