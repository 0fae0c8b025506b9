/* mv_oracle.c -- CPU restatement of the maveric-slam tracking hot path.
 * TEST INFRASTRUCTURE ONLY (see mv_oracle.h for the rules and the parity status).
 * Every function cites the reference file:line it restates; paths are relative to
 * the reference tree.  Compile with -fwrapv -ffp-contract=off (oracle/Makefile):
 * the reference overflows int32 at tracking_main.c:154 and that wrap is part of the
 * results; fp32 expressions must not be fused.
 */
#include "mv_oracle.h"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ===================================================================== */
/* Detector post-processing                                               */
/* ===================================================================== */

#define ORC_TAYLOR_TERMS 5 /* top_N.c:7  (#define P 5) */

/* top_N.c:59-63: {1, s/1, s^2/2!, ...} built by the recurrence c[i] = c[i-1]*s/i. */
static void taylor_coeffs(float scale, float c[ORC_TAYLOR_TERMS]) {
  c[0] = 1;
  for (int i = 1; i < ORC_TAYLOR_TERMS; i++) c[i] = c[i - 1] * scale / i;
}

/* top_N.c:12-20: 1 + sum_{i=1..4} c[i]*x^i with x^i kept in int32. */
static float taylor_exp(const float* c, int8_t x) {
  float acc = 1.0f;
  int xp = x;
  for (int i = 1; i < ORC_TAYLOR_TERMS; i++) {
    acc += c[i] * xp;
    xp *= x;
  }
  return acc;
}

/* top_N.c:22-49: softmax over the non-negative logits of one cell; argmax excludes
 * the dustbin (channel 64) but the dustbin is part of the denominator. */
static void cell_softmax(const float* c, const int8_t* row, int* best_ch, float* best_prob) {
  int arg = 64;
  float top = 0;
  float denom = FLT_MIN;
  for (int ch = 0; ch < 65; ch++) {
    if (row[ch] < 0) continue;
    float e = taylor_exp(c, row[ch]);
    if (ch != 64 && e > top) {
      top = e;
      arg = ch;
    }
    denom += e;
  }
  *best_ch = arg;
  *best_prob = top / denom;
}

/* top_N.c:136-165.  Returns the number of cells whose argmax is not the dustbin
 * (what the reference adds to *num_valid). */
int orc_softmax(float scale, const int8_t* semi, int cells, int* max_idx, float* probs) {
  float c[ORC_TAYLOR_TERMS];
  taylor_coeffs(scale, c);
  int valid = 0;
  for (int p = 0; p < cells; p++) {
    int arg;
    float pr;
    cell_softmax(c, semi + (size_t)p * 65, &arg, &pr);
    max_idx[p] = arg;
    if (arg != 64) {
      probs[p] = pr;
      valid++;
    } else {
      probs[p] = -1;
    }
  }
  return valid;
}

/* top_N.c:53-134.  Returns 1 where the reference prints "Exceed max number of
 * features!" and exits (top_N.c:91-94), else 0. */
int orc_top_n(float scale, const int8_t* semi, int cells, int N, int max_valid,
              int* num_selected, int* patches, int* indices, float* probs) {
  float c[ORC_TAYLOR_TERMS];
  taylor_coeffs(scale, c);
  *num_selected = 0;

  int* v_patch = (int*)malloc(sizeof(int) * (size_t)max_valid);
  int* v_idx = (int*)malloc(sizeof(int) * (size_t)max_valid);
  float* v_prob = (float*)malloc(sizeof(float) * (size_t)max_valid);
  float hi = 0, lo = FLT_MAX;
  int nv = 0;
  int overflow = 0;

  for (int p = 0; p < cells && !overflow; p++) {
    int arg = 64;
    float pr = -1;
    cell_softmax(c, semi + (size_t)p * 65, &arg, &pr);
    if (arg != 64 && pr > 0.01) { /* double compare, top_N.c:77 */
      v_patch[nv] = p;
      v_idx[nv] = arg;
      v_prob[nv] = pr;
      if (pr > hi) hi = pr;
      if (pr < lo) lo = pr;
      nv++;
      if (nv >= max_valid) overflow = 1;
    }
  }

  if (!overflow) {
    if (nv <= N) { /* top_N.c:98-106 */
      *num_selected = nv;
      for (int i = 0; i < nv; i++) {
        patches[i] = v_patch[i];
        indices[i] = v_idx[i];
        probs[i] = v_prob[i];
      }
    } else { /* top_N.c:108-133 */
      float split = N / (float)nv;
      float cut = hi * split + lo * (1 - split);
      int k = 0;
      for (int i = 0; i < nv && k < N; i++) {
        if (v_prob[i] >= cut) {
          patches[k] = v_patch[i];
          indices[k] = v_idx[i];
          probs[k] = v_prob[i];
          k++;
        }
      }
      *num_selected = k;
    }
  }
  free(v_patch);
  free(v_idx);
  free(v_prob);
  return overflow;
}

/* ===================================================================== */
/* Windowed int8 matcher                                                  */
/* ===================================================================== */

/* tracking_main.c:154.  `dot*dot` and `n_cand*n_query` are int32 products that wrap
 * (-fwrapv); the quotient is int -> float RN, then an IEEE fp32 divide. */
static float wrapped_cos2(int32_t dot, int32_t n_cand, int32_t n_query) {
  int32_t num = (int32_t)((uint32_t)dot * (uint32_t)dot);
  int32_t den = (int32_t)((uint32_t)n_cand * (uint32_t)n_query);
  return num / (float)den;
}

int orc_match(const orc_match_cfg* cfg, const int8_t* desc0, const int8_t* desc1,
              const int* max_idx0, const float* probs0,
              int nq, const int* patches1, const int* indices1,
              float* pts0, float* pts1, int* cell0, int* query, float* score,
              orc_match_stats* stats) {
  const int rows = cfg->rows, cols = cfg->cols, r = cfg->radius;
  const double accept = cfg->match_threshold * cfg->match_threshold; /* :155 */
  int n_out = 0;
  orc_match_stats st = {0, 0, 0};

  for (int i = 0; i < nq; i++) { /* :114 */
    const int cell1 = patches1[i];
    const int qx = cell1 / rows, qy = cell1 % rows; /* :59-62 */
    const int8_t* dq = desc1 + (size_t)cell1 * 256;

    /* :127-130, clamped inclusive window (frame-1 grid dims) */
    int x_lo = qx + cfg->shift_x - r; if (x_lo < 0) x_lo = 0;
    int x_hi = qx + cfg->shift_x + r; if (x_hi > cols - 1) x_hi = cols - 1;
    int y_lo = qy + cfg->shift_y - r; if (y_lo < 0) y_lo = 0;
    int y_hi = qy + cfg->shift_y + r; if (y_hi > rows - 1) y_hi = rows - 1;

    int32_t n_cand = 0; /* "norm1_squared": sticky candidate norm, :133 */
    int have = 0, best_ch = -1, best_x = 0, best_y = 0;
    float best = 0;

    for (int x = x_lo; x <= x_hi; x++) {   /* :135 */
      for (int y = y_lo; y <= y_hi; y++) { /* :136 */
        const int c = x * rows + y;        /* :64-66 */
        st.window_cells++;
        const int ch = max_idx0[c];
        if (ch == 64) continue;                  /* :142 */
        if (probs0[c] < cfg->min_prob0) continue; /* :146, double compare */
        const int8_t* dc = desc0 + (size_t)c * 256;

        /* :18-43 -- 256-d while the sticky candidate norm is zero, else 64-d with
         * the stale candidate norm and a 64-d query norm */
        int32_t dot = 0, n_query = 0;
        if (n_cand == 0) {
          for (int k = 0; k < 256; k++) {
            dot += dc[k] * dq[k];
            n_cand += dc[k] * dc[k];
            n_query += dq[k] * dq[k];
          }
          st.pairs_256++;
        } else {
          for (int k = 0; k < 64; k++) {
            dot += dc[k] * dq[k];
            n_query += dq[k] * dq[k];
          }
          st.pairs_64++;
        }
        const float s = wrapped_cos2(dot, n_cand, n_query);
        if (s > accept) {            /* :155 (float vs double) */
          if (!have || s > best) {   /* :156 strict: first wins ties */
            have = 1;
            best_ch = ch;
            best = s;
            best_x = x;
            best_y = y;
          }
        }
      }
    }

    if (have && n_out < cfg->max_matches) { /* :167-188 */
      const int ch1 = indices1[i];
      pts0[2 * n_out + 0] = (float)(best_x * 8 + best_ch % 8);
      pts0[2 * n_out + 1] = (float)(best_y * 8 + best_ch / 8);
      pts1[2 * n_out + 0] = (float)(qx * 8 + ch1 % 8);
      pts1[2 * n_out + 1] = (float)(qy * 8 + ch1 / 8);
      if (cell0) cell0[n_out] = best_x * rows + best_y;
      if (query) query[n_out] = i;
      if (score) score[n_out] = best;
      n_out++;
    }
    if (n_out >= cfg->max_matches) break; /* :190-192 */
  }
  if (stats) *stats = st;
  return n_out;
}

/* ===================================================================== */
/* 3x3 SVD (include/svd/svd.h: McAdams et al. TR1690 as implemented there) */
/* ===================================================================== */

static float bits_to_float(int32_t i) { float f; memcpy(&f, &i, 4); return f; }
static int32_t float_to_bits(float f) { int32_t i; memcpy(&i, &f, 4); return i; }

/* svd.h:37-48: magic-constant reciprocal square root, one Newton step. */
static float rsqrt_one_step(float x) {
  float half = 0.5f * x;
  float y = bits_to_float(0x5f375a82 - (float_to_bits(x) >> 1));
  return y * (1.5f - half * y * y);
}
/* svd.h:54-62: two Newton steps, different magic constant. */
static float rsqrt_two_steps(float x) {
  float half = 0.5f * x;
  float y = bits_to_float(0x5f37599e - (float_to_bits(x) >> 1));
  y = y * (1.5f - half * y * y);
  y = y * (1.5f - half * y * y);
  return y;
}

/* Symmetric 3x3 held as its lower triangle, in the rotating order svd.h uses. */
typedef struct { float d0, o10, d1, o20, o21, d2; } sym3;

/* svd.h:148-163 + :165-216: one approximate-Givens Jacobi step on the (0,1) block,
 * then the cyclic relabelling.  (ax, ay, az) is the axis triple of this step. */
static void jacobi_step(int ax, int ay, int az, sym3* s, float q[4]) {
  float ch = 2 * (s->d0 - s->d1);
  float sh = s->o10;
  /* 5.828427124 is a double literal in svd.h:22 -> the left side is double math */
  int keep = 5.828427124 * sh * sh < ch * ch;
  float w = rsqrt_one_step(ch * ch + sh * sh);
  ch = keep ? w * ch : (float)0.923879532;
  sh = keep ? w * sh : (float)0.3826834323;

  float nrm = ch * ch + sh * sh;
  float a = (ch * ch - sh * sh) / nrm;
  float b = (2 * sh * ch) / nrm;

  const float p00 = s->d0, p10 = s->o10, p11 = s->d1, p20 = s->o20, p21 = s->o21, p22 = s->d2;
  /* svd.h:185-187, S <- Q' S Q */
  float n00 = a * (a * p00 + b * p10) + b * (a * p10 + b * p11);
  float n10 = a * (-b * p00 + a * p10) + b * (-b * p10 + a * p11);
  float n11 = -b * (-b * p00 + a * p10) + a * (-b * p10 + a * p11);
  float n20 = a * p20 + b * p21;
  float n21 = -b * p20 + a * p21;
  float n22 = p22;

  /* svd.h:190-206, accumulate the rotation into the quaternion (x,y,z,w order) */
  float t0 = q[0] * sh, t1 = q[1] * sh, t2 = q[2] * sh;
  float tv[3] = {t0, t1, t2};
  sh *= q[3];
  q[0] *= ch; q[1] *= ch; q[2] *= ch; q[3] *= ch;
  q[az] += sh;
  q[3] -= tv[az];
  q[ax] += tv[ay];
  q[ay] -= tv[ax];

  /* svd.h:209-214, relabel so the next pivot block is again (0,1) */
  s->d0 = n11;
  s->o10 = n21; s->d1 = n22;
  s->o20 = n10; s->o21 = n20; s->d2 = n00;
}

static float sq3(float x, float y, float z) { return x * x + y * y + z * z; } /* svd.h:218 */

/* svd.h:77-83 applied to column pair (i,j) of a 3x3: X<-Y, Y<- -X when c. */
static void neg_swap_cols(int c, float M[3][3], int i, int j) {
  for (int r = 0; r < 3; r++) {
    float z = -M[r][i];
    M[r][i] = c ? M[r][j] : M[r][i];
    M[r][j] = c ? z : M[r][j];
  }
}

/* svd.h:277-291 */
static void qr_givens(float pivot, float below, float* ch, float* sh) {
  float eps = (float)1e-6;
  float sum = pivot * pivot + below * below;
  float rho = sum * rsqrt_two_steps(sum); /* svd.h:64-67 */
  float s = rho > eps ? below : 0;
  float c = fabsf(pivot) + fmaxf(rho, eps);
  if (pivot < 0) { float tmp = s; s = c; c = tmp; } /* svd.h:69-75 */
  float w = rsqrt_one_step(c * c + s * s);
  *ch = c * w;
  *sh = s * w;
}

/* svd.h:358-405.  S is the (approximately upper-triangular) R of the QR step. */
void orc_svd3(const float A[3][3], float U[3][3], float S[3][3], float V[3][3]) {
  /* A^T A, svd.h:117-119 (each entry a three-term left-to-right sum) */
  float ata[3][3];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++)
      ata[i][j] = A[0][i] * A[0][j] + A[1][i] * A[1][j] + A[2][i] * A[2][j];

  /* svd.h:226-244 */
  sym3 s = {ata[0][0], ata[1][0], ata[1][1], ata[2][0], ata[2][1], ata[2][2]};
  float q[4] = {0, 0, 0, 1};
  for (int sweep = 0; sweep < 4; sweep++) {
    jacobi_step(0, 1, 2, &s, q);
    jacobi_step(1, 2, 0, &s, q);
    jacobi_step(2, 0, 1, &s, q);
  }

  /* svd.h:122-146 */
  {
    float x = q[0], y = q[1], z = q[2], w = q[3];
    float xx = x * x, yy = y * y, zz = z * z, xz = x * z, xy = x * y, yz = y * z;
    float wx = w * x, wy = w * y, wz = w * z;
    V[0][0] = 1 - 2 * (yy + zz); V[0][1] = 2 * (xy - wz);     V[0][2] = 2 * (xz + wy);
    V[1][0] = 2 * (xy + wz);     V[1][1] = 1 - 2 * (xx + zz); V[1][2] = 2 * (yz - wx);
    V[2][0] = 2 * (xz - wy);     V[2][1] = 2 * (yz + wx);     V[2][2] = 1 - 2 * (xx + yy);
  }

  /* B = A V, svd.h:99-101 */
  float B[3][3];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++)
      B[i][j] = A[i][0] * V[0][j] + A[i][1] * V[1][j] + A[i][2] * V[2][j];

  /* svd.h:247-274: order columns by squared length, descending */
  {
    float r0 = sq3(B[0][0], B[1][0], B[2][0]);
    float r1 = sq3(B[0][1], B[1][1], B[2][1]);
    float r2 = sq3(B[0][2], B[1][2], B[2][2]);
    int c = r0 < r1;
    neg_swap_cols(c, B, 0, 1); neg_swap_cols(c, V, 0, 1);
    if (c) { float tmp = r0; r0 = r1; r1 = tmp; }
    c = r0 < r2;
    neg_swap_cols(c, B, 0, 2); neg_swap_cols(c, V, 0, 2);
    if (c) { float tmp = r0; r0 = r2; r2 = tmp; }
    c = r1 < r2;
    neg_swap_cols(c, B, 1, 2); neg_swap_cols(c, V, 1, 2);
  }

  /* svd.h:294-356: three Givens rotations */
  float ch1, sh1, ch2, sh2, ch3, sh3, a, b;
  float R[3][3], T[3][3];
  qr_givens(B[0][0], B[1][0], &ch1, &sh1);
  a = 1 - 2 * sh1 * sh1;
  b = 2 * ch1 * sh1;
  for (int j = 0; j < 3; j++) {
    R[0][j] = a * B[0][j] + b * B[1][j];
    R[1][j] = -b * B[0][j] + a * B[1][j];
    R[2][j] = B[2][j];
  }
  qr_givens(R[0][0], R[2][0], &ch2, &sh2);
  a = 1 - 2 * sh2 * sh2;
  b = 2 * ch2 * sh2;
  for (int j = 0; j < 3; j++) {
    T[0][j] = a * R[0][j] + b * R[2][j];
    T[1][j] = R[1][j];
    T[2][j] = -b * R[0][j] + a * R[2][j];
  }
  qr_givens(T[1][1], T[2][1], &ch3, &sh3);
  a = 1 - 2 * sh3 * sh3;
  b = 2 * ch3 * sh3;
  for (int j = 0; j < 3; j++) {
    S[0][j] = T[0][j];
    S[1][j] = a * T[1][j] + b * T[2][j];
    S[2][j] = -b * T[1][j] + a * T[2][j];
  }

  /* svd.h:341-355, Q = Q1 Q2 Q3 in closed form */
  float s1 = sh1 * sh1, s2 = sh2 * sh2, s3 = sh3 * sh3;
  U[0][0] = (-1 + 2 * s1) * (-1 + 2 * s2);
  U[0][1] = 4 * ch2 * ch3 * (-1 + 2 * s1) * sh2 * sh3 + 2 * ch1 * sh1 * (-1 + 2 * s3);
  U[0][2] = 4 * ch1 * ch3 * sh1 * sh3 - 2 * ch2 * (-1 + 2 * s1) * sh2 * (-1 + 2 * s3);
  U[1][0] = 2 * ch1 * sh1 * (1 - 2 * s2);
  U[1][1] = -8 * ch1 * ch2 * ch3 * sh1 * sh2 * sh3 + (-1 + 2 * s1) * (-1 + 2 * s3);
  U[1][2] = -2 * ch3 * sh3 + 4 * sh1 * (ch3 * sh1 * sh3 + ch1 * ch2 * sh2 * (-1 + 2 * s3));
  U[2][0] = 2 * ch2 * sh2;
  U[2][1] = 2 * ch3 * (1 - 2 * s2) * sh3;
  U[2][2] = (-1 + 2 * s2) * (-1 + 2 * s3);
}

/* ===================================================================== */
/* NMS between detector and matcher (src/run_nms.c:65-156)                 */
/* ===================================================================== */

/* Corners of the cell grid are visited x outer / y inner, both INCLUSIVE of the far edge
 * (:65-66).  Each corner looks at its (up to) four adjacent cells (:75-81) and takes the cell's
 * keypoint only if it lies within 6 px of the corner on both axes (:94-97).  Then, repeatedly:
 * the strongest remaining keypoint suppresses every other one closer than 4 px on both axes
 * (:131-147) and retires.  The first arg-max scan ignores patch 0 (`patches[i] > 0`, :116), the
 * second does not (:126) -- reproduced as written. */
int orc_nms(int rows, int cols, int* max_idx, float* probs1, int* events, int max_events) {
  int n_events = 0;
  for (int xi = 0; xi <= cols; xi++) {
    for (int yi = 0; yi <= rows; yi++) {
      int nv = 0, patches[4] = {0, 0, 0, 0}, xs[4] = {0, 0, 0, 0}, ys[4] = {0, 0, 0, 0};
      float probs[4] = {0, 0, 0, 0};
      for (int xd = -1; xd <= 0; xd++) {
        int xg = xi + xd;
        if (xg < 0 || xg >= cols) continue;
        for (int yd = -1; yd <= 0; yd++) {
          int yg = yi + yd;
          if (yg < 0 || yg >= rows) continue;
          int patch = xg * rows + yg;               /* grid_to_patch, :33-35 */
          int index = max_idx[patch];
          if (index == 64) continue;
          int px = index % 8, py = index / 8;       /* :37-40 */
          if (xd == -1 && px < 2) continue;
          if (xd == 0 && px >= 6) continue;
          if (yd == -1 && py < 2) continue;
          if (yd == 0 && py >= 6) continue;
          patches[nv] = patch; probs[nv] = probs1[patch];
          xs[nv] = xg * 8 + px; ys[nv] = yg * 8 + py;
          nv++;
        }
      }
      for (;;) {
        float max_prob = 0; int max_index = -1;
        for (int i = 0; i < nv; i++)
          if (patches[i] > 0 && probs[i] > max_prob) { max_prob = probs[i]; max_index = i; }
        if (max_index == -1) break;
        for (int i = 0; i < nv; i++)
          if (patches[i] >= 0 && probs[i] > max_prob) { max_prob = probs[i]; max_index = i; }
        for (int i = 0; i < nv; i++) {
          if (i == max_index || patches[i] < 0) continue;
          int xdiff = abs(xs[max_index] - xs[i]), ydiff = abs(ys[max_index] - ys[i]);
          if (xdiff < 4 && ydiff < 4) {
            max_idx[patches[i]] = 64;
            probs1[patches[i]] = 64;
            if (events && n_events < max_events) {
              events[4 * n_events] = xs[max_index]; events[4 * n_events + 1] = ys[max_index];
              events[4 * n_events + 2] = xs[i]; events[4 * n_events + 3] = ys[i];
            }
            n_events++;
            patches[i] = -1; probs[i] = -1;
          }
        }
        probs[max_index] = -1; patches[max_index] = -1;
      }
    }
  }
  return n_events;
}

/* ===================================================================== */
/* Essential-matrix RANSAC as the reference runs it (src/pnp_solver.c)    */
/* ===================================================================== */

/* pnp_solver.c:28-34 */
void orc_normalize_points(int n, const float* pts, const float K[3][3], float* out) {
  for (int i = 0; i < n; i++) {
    out[2 * i + 0] = (pts[2 * i + 0] - K[0][2]) / K[0][0];
    out[2 * i + 1] = (pts[2 * i + 1] - K[1][2]) / K[1][1];
  }
}

/* pnp_solver.c:89-105: || E [p1;1] - [p2;1] ||^2 (pixel units) */
float orc_reproj_error(const float p1[2], const float p2[2], const float E[3][3]) {
  const float h1[3] = {p1[0], p1[1], 1.0f};
  const float h2[3] = {p2[0], p2[1], 1.0f};
  float err = 0;
  for (int i = 0; i < 3; i++) {
    float proj = E[i][0] * h1[0] + E[i][1] * h1[1] + E[i][2] * h1[2];
    float d = proj - h2[i];
    err += d * d;
  }
  return err;
}

/* pnp_solver.c:110-165 with the model of :36-86, which is the identity for every
 * sample (:63 and :81-85), so the 8 rand() draws (:123) cannot change any output.
 * Returns 1 if some iteration found an inlier (outputs written), else 0 -- the
 * reference leaves best_E/num_inliers uninitialised in that case; here E = I and
 * *num_inliers = 0. */
int orc_ransac_identity(int n, const float* pts1, const float* pts2, int iters, float thr,
                        int cap, float best_E[3][3], int* best_inliers, int* num_inliers) {
  float E[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  int* tmp = (int*)malloc(sizeof(int) * (size_t)(cap > 0 ? cap : 1));
  int best = 0, wrote = 0;
  memcpy(best_E, E, sizeof(E));
  *num_inliers = 0;
  for (int it = 0; it < iters; it++) {
    int cnt = 0;
    for (int i = 0; i < n; i++) {
      float e = orc_reproj_error(pts1 + 2 * i, pts2 + 2 * i, E);
      if (e < thr && cnt < cap) tmp[cnt++] = i; /* :146 */
    }
    if (cnt > best || cnt == cap) { /* :152 */
      best = cnt;
      *num_inliers = cnt;
      memcpy(best_E, E, sizeof(E));
      if (best_inliers) memcpy(best_inliers, tmp, sizeof(int) * (size_t)cnt);
      wrote = 1;
    }
  }
  free(tmp);
  return wrote;
}

/* pnp_solver.c:168-194: R1 = U W, R2 = U W^T, t = U[:,2] */
void orc_recover_pose(const float E[3][3], float R1[3][3], float R2[3][3], float t[3]) {
  float U[3][3], S[3][3], V[3][3];
  orc_svd3(E, U, S, V);
  const float W[3][3] = {{0, -1, 0}, {1, 0, 0}, {0, 0, 1}};
  const float Wt[3][3] = {{0, 1, 0}, {-1, 0, 0}, {0, 0, 1}};
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      R1[i][j] = U[i][0] * W[0][j] + U[i][1] * W[1][j] + U[i][2] * W[2][j];
      R2[i][j] = U[i][0] * Wt[0][j] + U[i][1] * Wt[1][j] + U[i][2] * Wt[2][j];
    }
  for (int i = 0; i < 3; i++) t[i] = U[i][2];
}

/* ===================================================================== */
/* Geometry and the reprojection residual                                  */
/* ===================================================================== */

/* types.c:18-25, Hamilton product, (w,x,y,z) */
void orc_quat_mul(const float a[4], const float b[4], float o[4]) {
  o[0] = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  o[1] = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  o[2] = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  o[3] = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
}

/* types.c:62-73: (q (0,v) q*) + t, q not normalised */
void orc_apply_transform(const float pose[7], const float X[3], float out[3]) {
  const float q[4] = {pose[0], pose[1], pose[2], pose[3]};
  const float v[4] = {0, X[0], X[1], X[2]};
  const float qc[4] = {q[0], -q[1], -q[2], -q[3]};
  float qv[4], r[4];
  orc_quat_mul(q, v, qv);
  orc_quat_mul(qv, qc, r);
  out[0] = r[1] + 1 * pose[4];
  out[1] = r[2] + 1 * pose[5];
  out[2] = r[3] + 1 * pose[6];
}

/* projection_factor.c:12-33: cam_project(T X) - z */
void orc_projection_error(const float pose[7], const float X[3], const float z[2],
                          const float cam[4], float err[2]) {
  float Xc[3];
  orc_apply_transform(pose, X, Xc);
  float px = Xc[0] / Xc[2], py = Xc[1] / Xc[2];
  float u = px * cam[0] + cam[2];
  float v = py * cam[1] + cam[3];
  err[0] = u + -1 * z[0];
  err[1] = v + -1 * z[1];
}

/* ===================================================================== */
/* Matmul shim (include/gemmini_functions_cpu.h:14-56, 60-124)             */
/* ===================================================================== */

static void mm_accumulate(size_t I, size_t J, size_t K, const float* A, const float* B, float* C,
                          size_t sA, size_t sB, size_t sC, float as, float bs, int tA, int tB) {
  const size_t a_i = tA ? 1 : sA, a_k = tA ? sA : 1;
  const size_t b_k = tB ? 1 : sB, b_j = tB ? sB : 1;
  for (size_t i = 0; i < I; i++)
    for (size_t j = 0; j < J; j++) {
      float* c = C + i * sC + j;
      for (size_t k = 0; k < K; k++) *c += as * A[i * a_i + k * a_k] * bs * B[k * b_k + j * b_j];
    }
}

void orc_matmul(size_t I, size_t J, size_t K, const float* A, const float* B, float* C,
                size_t sA, size_t sB, size_t sC, float as, float bs, int tA, int tB) {
  mm_accumulate(I, J, K, A, B, C, sA, sB, sC, as, bs, tA, tB);
}

void orc_matmul2(size_t I, size_t J, size_t K, const float* A, const float* B,
                 const float* D, float* C, size_t sA, size_t sB, size_t sD, size_t sC,
                 float as, float bs, float ds, int tA, int tB) {
  if (D)
    for (size_t i = 0; i < I; i++)
      for (size_t j = 0; j < J; j++) C[i * sC + j] = ds * D[i * sD + j];
  mm_accumulate(I, J, K, A, B, C, sA, sB, sC, as, bs, tA, tB);
}

/* ===================================================================== */
/* Local bundle adjustment: Schur complement of the landmarks              */
/* (src/local_bundle_adjustment.c:133-246, SURVEY §8f rank 4)              */
/* ===================================================================== */

/* local_bundle_adjustment.c:48-75: cofactors over the determinant, each quotient on its own */
void orc_invert_3x3(float* matrix, int stride) {
  float m[9], inv[9];
  for (int j = 0; j < 3; j++)
    for (int i = 0; i < 3; i++) m[j * 3 + i] = matrix[j * stride + i];
  float det = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) +
              m[2] * (m[3] * m[7] - m[4] * m[6]);
  inv[0] = (m[4] * m[8] - m[5] * m[7]) / det;
  inv[1] = (m[2] * m[7] - m[1] * m[8]) / det;
  inv[2] = (m[1] * m[5] - m[2] * m[4]) / det;
  inv[3] = (m[5] * m[6] - m[3] * m[8]) / det;
  inv[4] = (m[0] * m[8] - m[2] * m[6]) / det;
  inv[5] = (m[2] * m[3] - m[0] * m[5]) / det;
  inv[6] = (m[3] * m[7] - m[4] * m[6]) / det;
  inv[7] = (m[1] * m[6] - m[0] * m[7]) / det;
  inv[8] = (m[0] * m[4] - m[1] * m[3]) / det;
  for (int j = 0; j < 3; j++)
    for (int i = 0; i < 3; i++) matrix[j * stride + i] = inv[j * 3 + i];
}

/* local_bundle_adjustment.c:35-46 with alpha = beta = 1, as every call site has it */
static void lba_add(const float* A, float* B, int rows, int cols, int sA, int sB) {
  for (int j = 0; j < cols; j++)
    for (int i = 0; i < rows; i++) B[j * sB + i] = 1.0f * A[j * sA + i] + 1.0f * B[j * sB + i];
}

/* The reduced camera matrix of one window: for every chunk of `chunk` landmarks, the factors'
 * [J|r]^T [J|r] blocks are scattered into the landmark block diagonal A, the pose-landmark block B
 * and the pose block C (:152-224), A is inverted block by block (:227), and C -= B A^-1 B^T
 * (:229-245).  C is (6 n_poses + 1)^2, column-major, its last row carrying J^T r (the last
 * column stays 0, as in the reference).
 *   J  [n_ldmks][n_poses][20]: the factor of (landmark, pose) as the reference stores it, a 2 x 10
 *      column-major block [dLandmark(3) | dPose(6) | residual(1)].
 * The reference's scratch persists across chunks and that is reproduced: off-diagonal blocks of A
 * stay 0, B A^-1 is overwritten as 0 * old + sum (so a non-finite entry sticks).  Its H_factor is
 * uninitialised stack before the first 0 * old; here it starts at 0.  n_ldmks % chunk == 0. */
void orc_lba_schur(int n_ldmks, int n_poses, int chunk, const float* J, float* C) {
  const int PD = 6 * n_poses, SH = PD + 1, LD = 3 * chunk;
  float* A = (float*)calloc((size_t)LD * LD, sizeof(float));
  float* B = (float*)calloc((size_t)SH * LD, sizeof(float));
  float* BA = (float*)calloc((size_t)SH * LD, sizeof(float));
  float H[100];
  memset(H, 0, sizeof(H));
  memset(C, 0, sizeof(float) * (size_t)SH * SH);
  for (int c0 = 0; c0 < n_ldmks; c0 += chunk) {
    for (int I = 0; I < LD; I += 3)                       /* :120-129 */
      for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) A[(I + i) * LD + I + j] = 0;
    memset(B, 0, sizeof(float) * (size_t)SH * LD);
    for (int ci = 0; ci < chunk; ci++) {
      for (int p = 0; p < n_poses; p++) {
        const int pi = p * 6, li = ci * 3;
        const float* Jf = J + ((size_t)(c0 + ci) * n_poses + p) * 20;
        orc_matmul2(10, 10, 2, Jf, Jf, H, H, 2, 2, 10, 10, 1, 1, 0, 0, 1);   /* :166-172 */
        lba_add(H, A + li * (LD + 1), 3, 3, 10, LD);                          /* H_LL :176-183 */
        lba_add(H + 3, B + pi + li * SH, 6, 3, 10, SH);                       /* H_PL :185-192 */
        lba_add(H + 9, B + (li + 1) * SH - 1, 1, 3, 10, SH);                  /* H_Lf :194-201 */
        lba_add(H + 33, C + pi * (SH + 1), 6, 6, 10, SH);                     /* H_PP :203-210 */
        lba_add(H + 39, C + (pi + 1) * SH - 1, 1, 6, 10, SH);                 /* H_Pf :212-219 */
      }
    }
    for (int I = 0; I < LD; I += 3) orc_invert_3x3(A + I * LD + I, LD);        /* :227 */
    orc_matmul2(LD, PD, LD, A, B, BA, BA, LD, SH, SH, SH, 1, 1, 0, 0, 0);      /* :230-235 */
    orc_matmul2(PD, PD, LD, B, BA, C, C, SH, SH, SH, SH, -1, 1, 1, 1, 0);      /* :238-243 */
  }
  free(A); free(B); free(BA);
}

/* The Gauss-Newton step of the reduced camera system: S d = -g with S the pose block of the
 * matrix orc_lba_schur returns and g its last row.  This is the cholesky() call the reference
 * leaves as a stub (local_bundle_adjustment.c:88-90,247), so it is THIS REPOSITORY'S DEFINITION
 * (PARITY UNPINNED): solve6() below, the 6 x 6 solve of the PnP kernel, for n = 6 n_poses --
 * diagonal s + damping * s + 1e-12, L L^T by rows with k ascending, forward substitution with k
 * ascending; only the back substitution runs k DESCENDING (n-1 ... i+1), the order in which a
 * column-oriented sweep meets the terms.  Only the lower triangle S[i][j], i >= j (C[j*SH + i])
 * is read.  Every sum is a chain of fmaf.  Returns 1 and d, or 0 and d = 0 when a pivot is not
 * positive (NaN included). */
int orc_lba_solve(int n_poses, float damping, const float* C, float* d) {
  const int n = 6 * n_poses, SH = n + 1;
  float* L = (float*)calloc((size_t)n * n, sizeof(float));
  float* inv = (float*)calloc((size_t)n, sizeof(float));
  float* y = (float*)calloc((size_t)n, sizeof(float));
  int ok = 1;
  for (int i = 0; i < n; i++) d[i] = 0.0f;
  for (int j = 0; j < n && ok; j++) {          /* column by column == row by row: same sums */
    for (int i = j; i < n; i++) {
      float s = C[(size_t)j * SH + i];
      if (i == j) s = fmaf(damping, s, s) + 1e-12f;
      for (int k = 0; k < j; k++) s = fmaf(-L[i * n + k], L[j * n + k], s);
      if (i == j) {
        if (!(s > 0.0f)) { ok = 0; break; }
        L[j * n + j] = sqrtf(s);
        inv[j] = 1.0f / L[j * n + j];
      } else {
        L[i * n + j] = s * inv[j];
      }
    }
  }
  if (ok) {
    for (int i = 0; i < n; i++) {
      float s = -C[(size_t)i * SH + n];
      for (int k = 0; k < i; k++) s = fmaf(-L[i * n + k], y[k], s);
      y[i] = s * inv[i];
    }
    for (int i = n - 1; i >= 0; i--) {
      float s = y[i];
      for (int k = n - 1; k > i; k--) s = fmaf(-L[k * n + i], d[k], s);
      d[i] = s * inv[i];
    }
  }
  free(L); free(inv); free(y);
  return ok;
}

/* ===================================================================== */
/* Counter-based random numbers shared by the generators and the sampler   */
/* ===================================================================== */

static uint64_t sm64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
static uint64_t ctr(uint64_t mixed_seed, uint64_t tag, uint64_t a, uint64_t b, uint64_t c) {
  return sm64(mixed_seed + ((tag << 56) | ((a & 0xFFFFFFull) << 32) | ((b & 0xFFFFFFull) << 8) |
                            (c & 0xFFull)));
}

/* ===================================================================== */
/* Gauss-Newton PnP RANSAC (PARITY UNPINNED: no reference implementation)  */
/* ===================================================================== */

typedef struct { float H[21], g[6], cost; int cnt; } ne_acc; /* upper triangle, row-major */

static void ne_zero(ne_acc* a) { memset(a, 0, sizeof(*a)); }

/* One correspondence into the normal equations.  Residual per projection_factor.c:
 * 27-33; Jacobian w.r.t. a left perturbation (omega, upsilon) of the pose. */
static void ne_add_point(ne_acc* acc, const float R[9], const float t[3], const orc_pnp_cfg* c,
                         float X, float Y, float Z, float u, float v, int gated) {
  float xc = fmaf(R[2], Z, fmaf(R[1], Y, fmaf(R[0], X, t[0])));
  float yc = fmaf(R[5], Z, fmaf(R[4], Y, fmaf(R[3], X, t[1])));
  float zc = fmaf(R[8], Z, fmaf(R[7], Y, fmaf(R[6], X, t[2])));
  int ok = zc > c->min_depth && zc < 1e30f;   /* depth gate: in front of the camera and finite */
  float iz = ok ? 1.0f / zc : 0.0f;
  float a = xc * iz, b = yc * iz;
  float ncu = c->cx - u, ncv = c->cy - v;   /* rounded once, when a correspondence is staged */
  float ru = fmaf(c->fx, a, ncu);
  float rv = fmaf(c->fy, b, ncv);
  float e2 = fmaf(rv, rv, ru * ru);
  int w = ok && (!gated || e2 < c->gate_sq);
  acc->cost += w ? e2 : 0.0f;
  acc->cnt += w;
  if (!w) return;   /* a correspondence that fails the gate contributes nothing */
  float fx = c->fx, fy = c->fy;
  float fxa = fx * a, fyb = fy * b, fiz = fx * iz, giz = fy * iz;
  float na = -a, nb = -b, nfy = -fy;
  float u0 = fxa * nb, u1 = fmaf(fxa, a, fx), u2 = fx * nb, u3 = fiz, u5 = fiz * na;
  float v0 = fmaf(fyb, nb, nfy), v1 = fyb * a, v2 = fy * a, v4 = giz, v5 = giz * nb;
  float* H = acc->H;
  /* row 0 */
  H[0] = fmaf(v0, v0, fmaf(u0, u0, H[0]));
  H[1] = fmaf(v0, v1, fmaf(u0, u1, H[1]));
  H[2] = fmaf(v0, v2, fmaf(u0, u2, H[2]));
  H[3] = fmaf(u0, u3, H[3]);
  H[4] = fmaf(v0, v4, H[4]);
  H[5] = fmaf(v0, v5, fmaf(u0, u5, H[5]));
  /* row 1 */
  H[6] = fmaf(v1, v1, fmaf(u1, u1, H[6]));
  H[7] = fmaf(v1, v2, fmaf(u1, u2, H[7]));
  H[8] = fmaf(u1, u3, H[8]);
  H[9] = fmaf(v1, v4, H[9]);
  H[10] = fmaf(v1, v5, fmaf(u1, u5, H[10]));
  /* row 2 */
  H[11] = fmaf(v2, v2, fmaf(u2, u2, H[11]));
  H[12] = fmaf(u2, u3, H[12]);
  H[13] = fmaf(v2, v4, H[13]);
  H[14] = fmaf(v2, v5, fmaf(u2, u5, H[14]));
  /* row 3 (H[16] = J3.J4 is structurally zero) */
  H[15] = fmaf(u3, u3, H[15]);
  H[17] = fmaf(u3, u5, H[17]);
  /* row 4 */
  H[18] = fmaf(v4, v4, H[18]);
  H[19] = fmaf(v4, v5, H[19]);
  /* row 5 */
  H[20] = fmaf(v5, v5, fmaf(u5, u5, H[20]));
  float* g = acc->g;
  g[0] = fmaf(v0, rv, fmaf(u0, ru, g[0]));
  g[1] = fmaf(v1, rv, fmaf(u1, ru, g[1]));
  g[2] = fmaf(v2, rv, fmaf(u2, ru, g[2]));
  g[3] = fmaf(u3, ru, g[3]);
  g[4] = fmaf(v4, rv, g[4]);
  g[5] = fmaf(v5, rv, fmaf(u5, ru, g[5]));
}

/* xor-butterfly over L lane partials, the order a shuffle reduction uses */
static void ne_butterfly(ne_acc lane[32], int L) {
  for (int off = L / 2; off >= 1; off >>= 1) {
    ne_acc nxt[32];
    for (int l = 0; l < L; l++) {
      for (int k = 0; k < 21; k++) nxt[l].H[k] = lane[l].H[k] + lane[l ^ off].H[k];
      for (int k = 0; k < 6; k++) nxt[l].g[k] = lane[l].g[k] + lane[l ^ off].g[k];
      nxt[l].cost = lane[l].cost + lane[l ^ off].cost;
      nxt[l].cnt = lane[l].cnt + lane[l ^ off].cnt;
    }
    memcpy(lane, nxt, sizeof(ne_acc) * (size_t)L);
  }
}

static void quat_to_R(const float q[4], float R[9]) {
  float w = q[0], x = q[1], y = q[2], z = q[3];
  float xx = x * x, yy = y * y, zz = z * z, xy = x * y, xz = x * z, yz = y * z;
  float wx = w * x, wy = w * y, wz = w * z;
  R[0] = 1.0f - 2.0f * (yy + zz); R[1] = 2.0f * (xy - wz);        R[2] = 2.0f * (xz + wy);
  R[3] = 2.0f * (xy + wz);        R[4] = 1.0f - 2.0f * (xx + zz); R[5] = 2.0f * (yz - wx);
  R[6] = 2.0f * (xz - wy);        R[7] = 2.0f * (yz + wx);        R[8] = 1.0f - 2.0f * (xx + yy);
}

static int tri(int i, int j) { /* index of (i,j), i<=j, in the packed upper triangle */
  return i * 6 - i * (i - 1) / 2 + (j - i);
}

/* Damped 6x6 Cholesky solve of H d = -g.  Returns 0 on a non-positive pivot. */
static int solve6(const ne_acc* acc, float damping, float d[6]) {
  float A[6][6], L[6][6], inv[6], y[6];
  for (int i = 0; i < 6; i++)
    for (int j = i; j < 6; j++) A[i][j] = A[j][i] = acc->H[tri(i, j)];
  for (int i = 0; i < 6; i++) A[i][i] = fmaf(damping, A[i][i], A[i][i]) + 1e-12f;
  for (int i = 0; i < 6; i++) {
    for (int j = 0; j <= i; j++) {
      float s = A[i][j];
      for (int k = 0; k < j; k++) s = fmaf(-L[i][k], L[j][k], s);
      if (i == j) {
        if (!(s > 0.0f)) return 0;
        L[i][i] = sqrtf(s);
        inv[i] = 1.0f / L[i][i];
      } else {
        L[i][j] = s * inv[j];
      }
    }
  }
  for (int i = 0; i < 6; i++) {
    float s = -acc->g[i];
    for (int k = 0; k < i; k++) s = fmaf(-L[i][k], y[k], s);
    y[i] = s * inv[i];
  }
  for (int i = 5; i >= 0; i--) {
    float s = y[i];
    for (int k = i + 1; k < 6; k++) s = fmaf(-L[k][i], d[k], s);
    d[i] = s * inv[i];
  }
  return 1;
}

/* pose <- Exp~(d) * pose with the Cayley-style retraction dq = normalise(1, w/2). */
static void retract(float q[4], float t[3], const float d[6]) {
  float hx = 0.5f * d[0], hy = 0.5f * d[1], hz = 0.5f * d[2];
  float n = 1.0f / sqrtf(fmaf(hz, hz, fmaf(hy, hy, fmaf(hx, hx, 1.0f))));
  float dq[4] = {n, hx * n, hy * n, hz * n};
  float dR[9];
  quat_to_R(dq, dR);
  float nt0 = fmaf(dR[2], t[2], fmaf(dR[1], t[1], dR[0] * t[0])) + d[3];
  float nt1 = fmaf(dR[5], t[2], fmaf(dR[4], t[1], dR[3] * t[0])) + d[4];
  float nt2 = fmaf(dR[8], t[2], fmaf(dR[7], t[1], dR[6] * t[0])) + d[5];
  t[0] = nt0; t[1] = nt1; t[2] = nt2;
  float nq[4];
  nq[0] = fmaf(-dq[3], q[3], fmaf(-dq[2], q[2], fmaf(-dq[1], q[1], dq[0] * q[0])));
  nq[1] = fmaf(-dq[3], q[2], fmaf(dq[2], q[3], fmaf(dq[1], q[0], dq[0] * q[1])));
  nq[2] = fmaf(dq[3], q[1], fmaf(dq[2], q[0], fmaf(-dq[1], q[3], dq[0] * q[2])));
  nq[3] = fmaf(dq[3], q[0], fmaf(-dq[2], q[1], fmaf(dq[1], q[2], dq[0] * q[3])));
  float m = 1.0f / sqrtf(fmaf(nq[3], nq[3], fmaf(nq[2], nq[2], fmaf(nq[1], nq[1], nq[0] * nq[0]))));
  q[0] = nq[0] * m; q[1] = nq[1] * m; q[2] = nq[2] * m; q[3] = nq[3] * m;
}

/* Accumulate over all n correspondences (gated) in the requested lane order. */
static void ne_all_points(ne_acc* out, const orc_pnp_cfg* c, const float R[9], const float t[3],
                          int n, int stride, const float* corr, int gated) {
  const float *PX = corr, *PY = corr + stride, *PZ = corr + 2 * stride, *PU = corr + 3 * stride,
              *PV = corr + 4 * stride;
  if (c->lanes > 1) {
    const int L = c->lanes;
    ne_acc lane[32];
    for (int l = 0; l < L; l++) {
      ne_zero(&lane[l]);
      for (int j = l; j < n; j += L)
        ne_add_point(&lane[l], R, t, c, PX[j], PY[j], PZ[j], PU[j], PV[j], gated);
    }
    ne_butterfly(lane, L);
    *out = lane[0];
  } else {
    ne_zero(out);
    for (int j = 0; j < n; j++) ne_add_point(out, R, t, c, PX[j], PY[j], PZ[j], PU[j], PV[j], gated);
  }
}

static void ne_sample_points(ne_acc* out, const orc_pnp_cfg* c, const float R[9], const float t[3],
                             int stride, const float* corr, const int* sample) {
  const float *PX = corr, *PY = corr + stride, *PZ = corr + 2 * stride, *PU = corr + 3 * stride,
              *PV = corr + 4 * stride;
  if (c->lanes > 1) {
    const int L = c->lanes;
    ne_acc lane[32];
    for (int l = 0; l < L; l++) {
      ne_zero(&lane[l]);
      for (int i = l; i < c->sample_size; i += L) {
        int j = sample[i];
        ne_add_point(&lane[l], R, t, c, PX[j], PY[j], PZ[j], PU[j], PV[j], 0);
      }
    }
    ne_butterfly(lane, L);
    *out = lane[0];
  } else {
    ne_zero(out);
    for (int i = 0; i < c->sample_size; i++) {
      int j = sample[i];
      ne_add_point(out, R, t, c, PX[j], PY[j], PZ[j], PU[j], PV[j], 0);
    }
  }
}

void orc_pnp_gn(const orc_pnp_cfg* c, int pair_index, int n, int stride, const float* corr,
                const float* init_pose, float* out_pose, float* out_stats, float* hyp_pose) {
  const float ident[7] = {1, 0, 0, 0, 0, 0, 0};
  const float* p0 = init_pose ? init_pose : ident;
  const uint64_t ms = sm64(c->seed);
  int best_h = -1, best_cnt = -1;
  float best_cost = 0, best_pose[7];
  memcpy(best_pose, p0, sizeof(best_pose));
  int sample[255];   /* mv_pnp_params_ok (pnp_gn.cu) accepts sample_size up to 255 */

  for (int h = 0; h < c->hypotheses && n > 0; h++) {
    float q[4] = {p0[0], p0[1], p0[2], p0[3]}, t[3] = {p0[4], p0[5], p0[6]};
    for (int i = 0; i < c->sample_size; i++) {
      uint64_t r = ctr(ms, 5, (uint64_t)pair_index, (uint64_t)h, (uint64_t)i);
      sample[i] = (int)(((r >> 32) * (uint64_t)n) >> 32);
    }
    int alive = 1;
    float R[9], d[6];
    ne_acc acc;
    for (int it = 0; it < c->sample_iters && alive; it++) {
      quat_to_R(q, R);
      ne_sample_points(&acc, c, R, t, stride, corr, sample);
      alive = solve6(&acc, c->damping, d);
      if (alive) retract(q, t, d);
    }
    for (int it = 0; it < c->refine_iters && alive; it++) {
      quat_to_R(q, R);
      ne_all_points(&acc, c, R, t, n, stride, corr, 1);
      alive = solve6(&acc, c->damping, d);
      if (alive) retract(q, t, d);
    }
    /* score under the final pose */
    quat_to_R(q, R);
    ne_all_points(&acc, c, R, t, n, stride, corr, 1);
    int cnt = alive ? acc.cnt : -1;
    float cost = acc.cost;
    if (hyp_pose) {
      float* o = hyp_pose + (size_t)h * 8;
      o[0] = q[0]; o[1] = q[1]; o[2] = q[2]; o[3] = q[3];
      o[4] = t[0]; o[5] = t[1]; o[6] = t[2]; o[7] = (float)cnt;
    }
    if (alive && (cnt > best_cnt || (cnt == best_cnt && cost < best_cost))) {
      best_cnt = cnt; best_cost = cost; best_h = h;
      best_pose[0] = q[0]; best_pose[1] = q[1]; best_pose[2] = q[2]; best_pose[3] = q[3];
      best_pose[4] = t[0]; best_pose[5] = t[1]; best_pose[6] = t[2];
    }
  }
  memcpy(out_pose, best_pose, sizeof(best_pose));
  out_stats[0] = (float)(best_cnt < 0 ? 0 : best_cnt);
  out_stats[1] = best_h < 0 ? 0.0f : best_cost;
  out_stats[2] = (float)best_h;
  out_stats[3] = best_h < 0 ? 0.0f : 1.0f;
}

/* ===================================================================== */
/* Synthetic KITTI-shaped frames                                           */
/* ===================================================================== */

static int8_t desc_lut(unsigned u) {
  static const int8_t tail[10] = {-128, -111, -97, -85, -70, 70, 85, 97, 111, 127};
  return u < 246 ? (int8_t)((int)(u % 67) - 33) : tail[u - 246];
}

void orc_synth_frame(const orc_synth_cfg* cfg, int frame, int off_x, int off_y,
                     int8_t* semi, int8_t* desc, float* depth) {
  const uint64_t ms = sm64(cfg->seed);
  const int rows = cfg->rows, cols = cfg->cols;
  const int amp = cfg->noise_amp;
  for (int x = 0; x < cols; x++)
    for (int y = 0; y < rows; y++) {
      const int cell = x * rows + y;
      const uint64_t wx = (uint64_t)(int64_t)(x + off_x + (1 << 23));
      const uint64_t wy = (uint64_t)(int64_t)(y + off_y + (1 << 23));
      const uint64_t k = ctr(ms, 1, wx, wy, 0);
      const int is_kp = (int)(k % 1000) < cfg->keypoint_permille;
      const int kp_ch = (int)((k >> 16) & 63);
      const int kp_val = 14 + (int)((k >> 24) % 29);
      const int kp_dust = -20 + (int)((k >> 32) % 45);
      const int bg_dust = 10 + (int)((k >> 32) % 30);
      if (depth) depth[cell] = 4.0f + (float)((k >> 40) & 0xFFFF) * (36.0f / 65536.0f);

      int8_t* srow = semi + (size_t)cell * 65;
      for (int g = 0; g < 9; g++) {
        uint64_t h = ctr(ms, 2, (uint64_t)frame, (uint64_t)cell, (uint64_t)g);
        for (int b = 0; b < 8; b++) {
          int ch = g * 8 + b;
          if (ch >= 65) break;
          unsigned u = (unsigned)((h >> (8 * b)) & 0xFF);
          int v = u == 255 ? (ch % 6) * 3 : -30 - (int)(u % 70);
          if (ch == 64) v = is_kp ? kp_dust : bg_dust;
          else if (is_kp && ch == kp_ch) v = kp_val;
          srow[ch] = (int8_t)v;
        }
      }

      int8_t* drow = desc + (size_t)cell * 256;
      for (int g = 0; g < 32; g++) {
        uint64_t hb = ctr(ms, 3, wx, wy, (uint64_t)g);
        uint64_t hn = ctr(ms, 4, (uint64_t)frame, (uint64_t)cell, (uint64_t)g);
        for (int b = 0; b < 8; b++) {
          int base = desc_lut((unsigned)((hb >> (8 * b)) & 0xFF));
          int noise = amp > 0 ? (int)(((hn >> (8 * b)) & 0xFF) % (unsigned)(2 * amp + 1)) - amp : 0;
          int v = base + noise;
          if (v > 127) v = 127;
          if (v < -128) v = -128;
          drow[g * 8 + b] = (int8_t)v;
        }
      }
    }
}

/* ===================================================================== */
/* Whole path for one frame pair (tracking_main.c:84-218 + GN-PnP)         */
/* ===================================================================== */

void orc_track_pair(const orc_track_cfg* cfg, int pair_index,
                    const int8_t* semi0, const int8_t* desc0, const float* depth0,
                    const int8_t* semi1, const int8_t* desc1, orc_pair_result* out) {
  const int cells = cfg->match.rows * cfg->match.cols;
  const int N = cfg->top_n, M = cfg->match.max_matches;
  int* max_idx0 = (int*)malloc(sizeof(int) * (size_t)cells);
  float* probs0 = (float*)malloc(sizeof(float) * (size_t)cells);
  int* qp = (int*)malloc(sizeof(int) * (size_t)N);
  int* qi = (int*)malloc(sizeof(int) * (size_t)N);
  float* qpr = (float*)malloc(sizeof(float) * (size_t)N);
  float* pts0 = (float*)malloc(sizeof(float) * 2 * (size_t)M);
  float* pts1 = (float*)malloc(sizeof(float) * 2 * (size_t)M);
  int* cell0 = (int*)malloc(sizeof(int) * (size_t)M);
  float* corr = (float*)malloc(sizeof(float) * 5 * (size_t)M);
  int* inl = (int*)malloc(sizeof(int) * (size_t)M);
  memset(out, 0, sizeof(*out));

  orc_softmax(cfg->semi_scale, semi0, cells, max_idx0, probs0); /* tracking_main.c:85-90 */
  int nq = 0;
  int overflow = orc_top_n(cfg->semi_scale, semi1, cells, N, cfg->max_valid, &nq, qp, qi, qpr);
  out->status = overflow ? 4 : 0;
  int nm = overflow ? 0 : orc_match(&cfg->match, desc0, desc1, max_idx0, probs0, nq, qp, qi,
                                    pts0, pts1, cell0, NULL, NULL, NULL);
  out->num_matches = nm;

  if (cfg->ransac_iters > 0) { /* tracking_main.c:199-218 */
    float E[3][3];
    int ninl = 0;
    /* the reference's inlier array holds MAX_NUM_INLIERS = 1000 entries (pnp_solver.c:107,:146) */
    orc_ransac_identity(nm, pts0, pts1, cfg->ransac_iters, cfg->ransac_thr, M < 1000 ? M : 1000, E, inl, &ninl);
    out->ransac_inliers = ninl;
  }

  /* landmarks: X = depth * K^-1 (x0, y0, 1) */
  for (int j = 0; j < nm; j++) {
    float d = depth0[cell0[j]];
    corr[0 * M + j] = (pts0[2 * j] - cfg->pnp.cx) / cfg->pnp.fx * d;
    corr[1 * M + j] = (pts0[2 * j + 1] - cfg->pnp.cy) / cfg->pnp.fy * d;
    corr[2 * M + j] = d;
    corr[3 * M + j] = pts1[2 * j];
    corr[4 * M + j] = pts1[2 * j + 1];
  }
  float pose[7], stats[4];
  orc_pnp_gn(&cfg->pnp, pair_index, nm, M, corr, NULL, pose, stats, NULL);
  memcpy(out->q, pose, 16);
  memcpy(out->t, pose + 4, 12);
  out->pnp_inliers = stats[0];
  out->pnp_cost = stats[1];
  out->best_h = (int)stats[2];

  free(max_idx0); free(probs0); free(qp); free(qi); free(qpr);
  free(pts0); free(pts1); free(cell0); free(corr); free(inl);
}

/* ------------------------------------------------------------------------------------------
 * BoW word assignment -- src/bow_main.c:13-55 (helpers, followed line for line) and :62-125 (the stated
 * definition of mv_oracle.h; the program itself has no defined result)
 * ------------------------------------------------------------------------------------------ */
void orc_bow_binarize(float scale, const int8_t* feature, int* binary8) {
  for (int i = 0; i < 8; i++) {               /* bow_main.c:13-41 with size = 8 */
    unsigned w = 0;
    for (int j = 0; j < 32; j++) {
      const int v = feature[i * 32 + j];
      w <<= 1;
      if (scale > 0 ? (v > 0) : (v <= 0)) w += 1;   /* :21 / :33 */
    }
    binary8[i] = (int)w;
  }
}

int orc_bow_matching_bits(const int* a, const int* b, int size) {
  int count = 0;                              /* bow_main.c:43-55: popcount of ~(a ^ b), byte by byte */
  for (int i = 0; i < size; i++) {
    unsigned m = ~((unsigned)a[i] ^ (unsigned)b[i]);
    while (m) { count += (int)(m & 1u); m >>= 1; }
  }
  return count;
}

void orc_bow_assign(const orc_bow_vocab* v, float desc_scale, const int8_t* desc, int* base, int* wid) {
  int sel = 0;                                /* :89 sel_base_nodes[i] = 0 */
  float max_score = 0.0f;                     /* :91 */
  for (int j = 0; j < v->n_base; j++) {
    int raw = 0;
    for (int k = 0; k < 256; k++) raw += (int)desc[k] * (int)v->base_desc[k * v->n_base + j];
    float m = rintf(desc_scale * (float)raw * (1.0f / 256.0f));
    if (m > 127.0f) m = 127.0f;
    if (m < -128.0f) m = -128.0f;
    if (m != m) m = 0.0f;
    const float score = v->scale[j] * m + 256.0f * v->bias[j];   /* :94, unfused */
    if (score > max_score) { max_score = score; sel = j; }       /* :96-99 */
  }
  int bits[8];
  orc_bow_binarize(desc_scale, desc, bits);
  int best_match = 0, best_wid = 0;           /* :108-109 */
  for (int w = 0; w < v->words_per_base; w++) {
    const int match = orc_bow_matching_bits(bits, v->leaves + ((size_t)sel * v->words_per_base + w) * 4, 8);   /* :111 */
    if (match > best_match) { best_match = match; best_wid = w; }   /* :112-115 */
  }
  *base = sel;
  *wid = best_wid;
}

/* ------------------------------------------------------------------------------------------
 * landmark table: local_feature_pool.h:24-62 applied per word id (the hash table's slot layout is not
 * part of the contents)
 * ------------------------------------------------------------------------------------------ */
void orc_pool_observe(orc_local_feature* table, int n_words, int frame, int n, const int* word_ids, const float* coords) {
  for (int i = 0; i < n; i++) {               /* local_feature_matching.c:153-161 */
    const int w = word_ids[i];
    if (w < 0 || w >= n_words) continue;
    orc_local_feature* f = &table[w];
    if (f->word_id == -1) {                   /* inserted: init_local_feature_with_id, :31-36 */
      f->word_id = w; f->frame_ptr = 0; f->num_frames = 1; f->frames[0] = frame;
      for (int c = 0; c < 3; c++) f->coords[c] = coords ? coords[3 * i + c] : 0.0f;
    } else if (f->num_frames < 8) {           /* update_local_feature, :38-48 */
      f->frames[(f->frame_ptr + f->num_frames) % 8] = frame;
      f->num_frames++;
    } else {
      f->frames[f->frame_ptr] = frame;
      f->frame_ptr = (f->frame_ptr + 1) % 8;
    }
  }
}

void orc_pool_remove_old(orc_local_feature* table, int n_words, int current_frame) {
  const int keep = current_frame - 8 + 1;     /* local_feature_pool.h:268-279 with remove_old_frame :50-62 */
  for (int w = 0; w < n_words; w++) {
    orc_local_feature* f = &table[w];
    if (f->word_id == -1) continue;
    if (f->frames[f->frame_ptr] < keep) {
      f->frame_ptr = (f->frame_ptr + 1) % 8;
      f->num_frames--;
    }
    if (f->num_frames == 0) { f->word_id = -1; f->frame_ptr = 0; f->num_frames = 0; }   /* delete_hash_entry */
  }
}

static double now_s(void) {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

double orc_bench_sequence(const orc_track_cfg* cfg, const orc_synth_cfg* syn, const int* offsets,
                          int first, int n, int threads, orc_pair_result* out) {
  const int cells = syn->rows * syn->cols;
  const int nf = n + 1;
  int8_t* semi = (int8_t*)malloc((size_t)nf * cells * 65);
  int8_t* desc = (int8_t*)malloc((size_t)nf * cells * 256);
  float* depth = (float*)malloc(sizeof(float) * (size_t)nf * cells);
#ifdef _OPENMP
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
#endif
  for (int f = 0; f < nf; f++)
    orc_synth_frame(syn, first + f, offsets[2 * f], offsets[2 * f + 1],
                    semi + (size_t)f * cells * 65, desc + (size_t)f * cells * 256,
                    depth + (size_t)f * cells);
  double t0 = now_s();
#ifdef _OPENMP
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
#endif
  for (int p = 0; p < n; p++)
    orc_track_pair(cfg, first + p, semi + (size_t)p * cells * 65, desc + (size_t)p * cells * 256,
                   depth + (size_t)p * cells, semi + (size_t)(p + 1) * cells * 65,
                   desc + (size_t)(p + 1) * cells * 256, &out[p]);
  double t1 = now_s();
  (void)threads;
  free(semi); free(desc); free(depth);
  return t1 - t0;
}
