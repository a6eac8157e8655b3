/* lbfgsb.c -- L-BFGS-B 3.0, the limited-memory quasi-Newton method for bound-constrained
 * minimisation, behind the reverse-communication entry point setulb().
 *
 * Algorithm: R. H. Byrd, P. Lu, J. Nocedal and C. Zhu, "A limited memory algorithm for bound
 * constrained optimization", SIAM J. Sci. Comput. 16 (1995) 1190-1208; C. Zhu, R. H. Byrd,
 * P. Lu and J. Nocedal, "Algorithm 778: L-BFGS-B", ACM TOMS 23 (1997) 550-560; version 3.0
 * with the subspace step of J. L. Morales and J. Nocedal, ACM TOMS 38 (2011) 7.  The line
 * search is the one of J. J. More and D. J. Thuente, ACM TOMS 20 (1994) 286-307 (MINPACK-2
 * dcsrch / dcstep).
 *
 * The interface is the one of the C translation of version 3.0 that RootDigger links: integer
 * task codes (START = 1, NEW_X = 2, FG = 10..15, ...), `logical` is int, and the workspace
 * sizes are wa[2mn + 5n + 11m^2 + 8m], iwa[3n], lsave[4], isave[44], dsave[29].  The arithmetic
 * follows the published Fortran statement by statement (the BLAS sums run in index order, as the
 * reference BLAS does), so that a caller sees the same iterates.  Nothing is printed: iprint is
 * accepted for the interface and otherwise ignored.
 *
 * Arrays are column-major and indexed from 1 through the macros below, as in the Fortran. */
#include <float.h>
#include <math.h>
#include <string.h>

/* task codes */
enum {
  START = 1, NEW_X = 2, ABNORMAL = 3, RESTART = 4,
  FG = 10, FG_LN = 11, FG_ST = 12, FG_END = 15,
  CONV_GRAD = 21, CONV_F = 22,
  STOP = 30, STOP_CPU = 31, STOP_END = 40,
  WARNING_ROUND = 101, WARNING_XTOL = 102, WARNING_STPMAX = 103, WARNING_STPMIN = 104,
  ERROR_SMALLSTP = 201, ERROR_LARGESTP = 202, ERROR_INITIAL_G = 203, ERROR_FTOL = 204, ERROR_GTOL = 205,
  ERROR_XTOL = 206, ERROR_STP0 = 207, ERROR_STP1 = 208, ERROR_N0 = 209, ERROR_M0 = 210, ERROR_FACTR = 211,
  ERROR_NBD = 212, ERROR_FEAS = 213
};
#define IS_FG(t) ((t) >= FG && (t) <= FG_END)
#define IS_STOP(t) ((t) >= STOP && (t) <= STOP_END)
#define IS_ERROR(t) ((t) >= 200 && (t) < 300)

/* dcsrch task codes (kept in csave) */
enum { LS_START = 1, LS_FG = 10, LS_CONV = 20, LS_WARN = 100, LS_ERROR = 200 };

/* ---------------------------------------------------------------------------------------------
 * BLAS level 1 (unit stride) and LINPACK
 * ------------------------------------------------------------------------------------------- */
static double ddot(int n, const double *x, const double *y) {
  double s = 0.0;
  for (int i = 0; i < n; ++i) s = s + x[i] * y[i];
  return s;
}
static void daxpy(int n, double a, const double *x, double *y) {
  for (int i = 0; i < n; ++i) y[i] = y[i] + a * x[i];
}
static void dscal(int n, double a, double *x) {
  for (int i = 0; i < n; ++i) x[i] = a * x[i];
}
static void dcopy(int n, const double *x, double *y) {
  for (int i = 0; i < n; ++i) y[i] = x[i];
}

/* Cholesky factor of the n x n leading block of a (leading dimension lda), R'R with R in the
 * upper triangle; info = 0, or the order of the leading minor that is not positive definite */
static void dpofa(double *a, int lda, int n, int *info) {
#define A(i, j) a[((j)-1) * (size_t)lda + (i)-1]
  for (int j = 1; j <= n; ++j) {
    *info = j;
    double s = 0.0;
    for (int k = 1; k <= j - 1; ++k) {
      double t = A(k, j) - ddot(k - 1, &A(1, k), &A(1, j));
      t = t / A(k, k);
      A(k, j) = t;
      s = s + t * t;
    }
    s = A(j, j) - s;
    if (s <= 0.0) return;
    A(j, j) = sqrt(s);
  }
  *info = 0;
#undef A
}

/* triangular solve, LINPACK job codes: 00 T x = b (T lower), 01 T x = b (T upper),
 * 10 T' x = b (T lower), 11 T' x = b (T upper); info = index of a zero diagonal element, or 0 */
static void dtrsl(const double *t, int ldt, int n, double *b, int job, int *info) {
#define T(i, j) t[((j)-1) * (size_t)ldt + (i)-1]
#define B(i) b[(i)-1]
  for (*info = 1; *info <= n; ++*info)
    if (T(*info, *info) == 0.0) return;
  *info = 0;
  int kase = 1;
  if (job % 10 != 0) kase = 2;
  if ((job % 100) / 10 != 0) kase += 2;
  switch (kase) {
    case 1:
      B(1) = B(1) / T(1, 1);
      for (int j = 2; j <= n; ++j) {
        daxpy(n - j + 1, -B(j - 1), &T(j, j - 1), &B(j));
        B(j) = B(j) / T(j, j);
      }
      break;
    case 2:
      B(n) = B(n) / T(n, n);
      for (int jj = 2; jj <= n; ++jj) {
        int j = n - jj + 1;
        daxpy(j, -B(j + 1), &T(1, j + 1), &B(1));
        B(j) = B(j) / T(j, j);
      }
      break;
    case 3:
      B(n) = B(n) / T(n, n);
      for (int jj = 2; jj <= n; ++jj) {
        int j = n - jj + 1;
        B(j) = B(j) - ddot(jj - 1, &T(j + 1, j), &B(j + 1));
        B(j) = B(j) / T(j, j);
      }
      break;
    default:
      B(1) = B(1) / T(1, 1);
      for (int j = 2; j <= n; ++j) {
        B(j) = B(j) - ddot(j - 1, &T(1, j), &B(1));
        B(j) = B(j) / T(j, j);
      }
      break;
  }
#undef T
#undef B
}

/* ---------------------------------------------------------------------------------------------
 * The line search: More & Thuente (MINPACK-2 dcsrch / dcstep)
 * ------------------------------------------------------------------------------------------- */
static double dmax3(double a, double b, double c) { return fmax(fmax(a, b), c); }

static void dcstep(double *stx, double *fx, double *dx, double *sty, double *fy, double *dy, double *stp,
                   double fp, double dp, int *brackt, double stpmin, double stpmax) {
  const double p66 = 0.66, two = 2.0, three = 3.0;
  double theta, s, gamma, p, q, r, stpc, stpq, stpf;
  const double sgnd = dp * (*dx / fabs(*dx));

  if (fp > *fx) {
    theta = three * (*fx - fp) / (*stp - *stx) + *dx + dp;
    s = dmax3(fabs(theta), fabs(*dx), fabs(dp));
    gamma = s * sqrt((theta / s) * (theta / s) - (*dx / s) * (dp / s));
    if (*stp < *stx) gamma = -gamma;
    p = (gamma - *dx) + theta;
    q = ((gamma - *dx) + gamma) + dp;
    r = p / q;
    stpc = *stx + r * (*stp - *stx);
    stpq = *stx + ((*dx / ((*fx - fp) / (*stp - *stx) + *dx)) / two) * (*stp - *stx);
    if (fabs(stpc - *stx) < fabs(stpq - *stx))
      stpf = stpc;
    else
      stpf = stpc + (stpq - stpc) / two;
    *brackt = 1;
  } else if (sgnd < 0.0) {
    theta = three * (*fx - fp) / (*stp - *stx) + *dx + dp;
    s = dmax3(fabs(theta), fabs(*dx), fabs(dp));
    gamma = s * sqrt((theta / s) * (theta / s) - (*dx / s) * (dp / s));
    if (*stp > *stx) gamma = -gamma;
    p = (gamma - dp) + theta;
    q = ((gamma - dp) + gamma) + *dx;
    r = p / q;
    stpc = *stp + r * (*stx - *stp);
    stpq = *stp + (dp / (dp - *dx)) * (*stx - *stp);
    if (fabs(stpc - *stp) > fabs(stpq - *stp))
      stpf = stpc;
    else
      stpf = stpq;
    *brackt = 1;
  } else if (fabs(dp) < fabs(*dx)) {
    theta = three * (*fx - fp) / (*stp - *stx) + *dx + dp;
    s = dmax3(fabs(theta), fabs(*dx), fabs(dp));
    gamma = s * sqrt(fmax(0.0, (theta / s) * (theta / s) - (*dx / s) * (dp / s)));
    if (*stp > *stx) gamma = -gamma;
    p = (gamma - dp) + theta;
    q = (gamma + (*dx - dp)) + gamma;
    r = p / q;
    if (r < 0.0 && gamma != 0.0)
      stpc = *stp + r * (*stx - *stp);
    else if (*stp > *stx)
      stpc = stpmax;
    else
      stpc = stpmin;
    stpq = *stp + (dp / (dp - *dx)) * (*stx - *stp);
    if (*brackt) {
      if (fabs(stpc - *stp) < fabs(stpq - *stp))
        stpf = stpc;
      else
        stpf = stpq;
      if (*stp > *stx)
        stpf = fmin(*stp + p66 * (*sty - *stp), stpf);
      else
        stpf = fmax(*stp + p66 * (*sty - *stp), stpf);
    } else {
      if (fabs(stpc - *stp) > fabs(stpq - *stp))
        stpf = stpc;
      else
        stpf = stpq;
      stpf = fmin(stpmax, stpf);
      stpf = fmax(stpmin, stpf);
    }
  } else {
    if (*brackt) {
      theta = three * (fp - *fy) / (*sty - *stp) + *dy + dp;
      s = dmax3(fabs(theta), fabs(*dy), fabs(dp));
      gamma = s * sqrt((theta / s) * (theta / s) - (*dy / s) * (dp / s));
      if (*stp > *sty) gamma = -gamma;
      p = (gamma - dp) + theta;
      q = ((gamma - dp) + gamma) + *dy;
      r = p / q;
      stpc = *stp + r * (*sty - *stp);
      stpf = stpc;
    } else if (*stp > *stx) {
      stpf = stpmax;
    } else {
      stpf = stpmin;
    }
  }

  if (fp > *fx) {
    *sty = *stp;
    *fy = fp;
    *dy = dp;
  } else {
    if (sgnd < 0.0) {
      *sty = *stx;
      *fy = *fx;
      *dy = *dx;
    }
    *stx = *stp;
    *fx = fp;
    *dx = dp;
  }
  *stp = stpf;
}

/* isave[0..1] and dsave[0..12] hold the search's state between calls */
static void dcsrch(double f, double g, double *stp, double ftol, double gtol, double xtol, double stpmin,
                   double stpmax, int *task, int *isave, double *dsave) {
  const double p5 = 0.5, p66 = 0.66, xtrapl = 1.1, xtrapu = 4.0;
  int    brackt, stage;
  double ginit, gtest, gx, gy, finit, fx, fy, stx, sty, stmin, stmax, width, width1, ftest;

  if (*task == LS_START) {
    if (*stp < stpmin) *task = LS_ERROR + 1;
    if (*stp > stpmax) *task = LS_ERROR + 2;
    if (g >= 0.0) *task = LS_ERROR + 3;
    if (ftol < 0.0) *task = LS_ERROR + 4;
    if (gtol < 0.0) *task = LS_ERROR + 5;
    if (xtol < 0.0) *task = LS_ERROR + 6;
    if (stpmin < 0.0) *task = LS_ERROR + 7;
    if (stpmax < stpmin) *task = LS_ERROR + 8;
    if (*task >= LS_ERROR) return;
    brackt = 0;
    stage = 1;
    finit = f;
    ginit = g;
    gtest = ftol * ginit;
    width = stpmax - stpmin;
    width1 = width / p5;
    stx = 0.0;
    fx = finit;
    gx = ginit;
    sty = 0.0;
    fy = finit;
    gy = ginit;
    stmin = 0.0;
    stmax = *stp + xtrapu * *stp;
    *task = LS_FG;
    goto save;
  }
  brackt = isave[0];
  stage = isave[1];
  ginit = dsave[0];
  gtest = dsave[1];
  gx = dsave[2];
  gy = dsave[3];
  finit = dsave[4];
  fx = dsave[5];
  fy = dsave[6];
  stx = dsave[7];
  sty = dsave[8];
  stmin = dsave[9];
  stmax = dsave[10];
  width = dsave[11];
  width1 = dsave[12];

  ftest = finit + *stp * gtest;
  if (stage == 1 && f <= ftest && g >= 0.0) stage = 2;
  if (brackt && (*stp <= stmin || *stp >= stmax)) *task = LS_WARN + 1;
  if (brackt && stmax - stmin <= xtol * stmax) *task = LS_WARN + 2;
  if (*stp == stpmax && f <= ftest && g <= gtest) *task = LS_WARN + 3;
  if (*stp == stpmin && (f > ftest || g >= gtest)) *task = LS_WARN + 4;
  if (f <= ftest && fabs(g) <= gtol * (-ginit)) *task = LS_CONV;
  if (*task == LS_CONV || (*task >= LS_WARN && *task < LS_ERROR)) goto save;

  if (stage == 1 && f <= fx && f > ftest) {
    double fm = f - *stp * gtest, fxm = fx - stx * gtest, fym = fy - sty * gtest;
    double gm = g - gtest, gxm = gx - gtest, gym = gy - gtest;
    dcstep(&stx, &fxm, &gxm, &sty, &fym, &gym, stp, fm, gm, &brackt, stmin, stmax);
    fx = fxm + stx * gtest;
    fy = fym + sty * gtest;
    gx = gxm + gtest;
    gy = gym + gtest;
  } else {
    dcstep(&stx, &fx, &gx, &sty, &fy, &gy, stp, f, g, &brackt, stmin, stmax);
  }
  if (brackt) {
    if (fabs(sty - stx) >= p66 * width1) *stp = stx + p5 * (sty - stx);
    width1 = width;
    width = fabs(sty - stx);
  }
  if (brackt) {
    stmin = fmin(stx, sty);
    stmax = fmax(stx, sty);
  } else {
    stmin = *stp + xtrapl * (*stp - stx);
    stmax = *stp + xtrapu * (*stp - stx);
  }
  *stp = fmax(*stp, stpmin);
  *stp = fmin(*stp, stpmax);
  if ((brackt && (*stp <= stmin || *stp >= stmax)) || (brackt && stmax - stmin <= xtol * stmax)) *stp = stx;
  *task = LS_FG;

save:
  isave[0] = brackt;
  isave[1] = stage;
  dsave[0] = ginit;
  dsave[1] = gtest;
  dsave[2] = gx;
  dsave[3] = gy;
  dsave[4] = finit;
  dsave[5] = fx;
  dsave[6] = fy;
  dsave[7] = stx;
  dsave[8] = sty;
  dsave[9] = stmin;
  dsave[10] = stmax;
  dsave[11] = width;
  dsave[12] = width1;
}

/* ---------------------------------------------------------------------------------------------
 * The pieces of one iteration
 * ------------------------------------------------------------------------------------------- */
#define X1(v, i) (v)[(i)-1]
#define WS(i, j) ws[((j)-1) * (size_t)n + (i)-1]
#define WY(i, j) wy[((j)-1) * (size_t)n + (i)-1]
#define SY(i, j) sy[((j)-1) * (size_t)m + (i)-1]
#define SS(i, j) ss[((j)-1) * (size_t)m + (i)-1]
#define WT(i, j) wt[((j)-1) * (size_t)m + (i)-1]
#define WN(i, j) wn[((j)-1) * (size_t)(2 * m) + (i)-1]
#define WN1(i, j) wn1[((j)-1) * (size_t)(2 * m) + (i)-1]

/* project x onto the box, classify the variables (iwhere: -1 free, 3 fixed, 0 otherwise) */
static void active(int n, const double *l, const double *u, const int *nbd, double *x, int *iwhere, int *prjctd,
                   int *cnstnd, int *boxed) {
  *prjctd = 0;
  *cnstnd = 0;
  *boxed = 1;
  for (int i = 1; i <= n; ++i) {
    if (X1(nbd, i) > 0) {
      if (X1(nbd, i) <= 2 && X1(x, i) <= X1(l, i)) {
        if (X1(x, i) < X1(l, i)) {
          *prjctd = 1;
          X1(x, i) = X1(l, i);
        }
      } else if (X1(nbd, i) >= 2 && X1(x, i) >= X1(u, i)) {
        if (X1(x, i) > X1(u, i)) {
          *prjctd = 1;
          X1(x, i) = X1(u, i);
        }
      }
    }
  }
  for (int i = 1; i <= n; ++i) {
    if (X1(nbd, i) != 2) *boxed = 0;
    if (X1(nbd, i) == 0) {
      X1(iwhere, i) = -1;
    } else {
      *cnstnd = 1;
      if (X1(nbd, i) == 2 && X1(u, i) - X1(l, i) <= 0.0)
        X1(iwhere, i) = 3;
      else
        X1(iwhere, i) = 0;
    }
  }
}

/* p := M v for the 2col x 2col middle matrix M of the compact L-BFGS form */
static void bmv(int m, const double *sy, const double *wt, int col, const double *v, double *p, int *info) {
  if (col == 0) return;
  X1(p, col + 1) = X1(v, col + 1);
  for (int i = 2; i <= col; ++i) {
    int    i2 = col + i;
    double sum = 0.0;
    for (int k = 1; k <= i - 1; ++k) sum = sum + SY(i, k) * X1(v, k) / SY(k, k);
    X1(p, i2) = X1(v, i2) + sum;
  }
  dtrsl(wt, m, col, &X1(p, col + 1), 11, info);
  if (*info != 0) return;
  for (int i = 1; i <= col; ++i) X1(p, i) = X1(v, i) / sqrt(SY(i, i));
  dtrsl(wt, m, col, &X1(p, col + 1), 1, info);
  if (*info != 0) return;
  for (int i = 1; i <= col; ++i) X1(p, i) = -X1(p, i) / sqrt(SY(i, i));
  for (int i = 1; i <= col; ++i) {
    double sum = 0.0;
    for (int k = i + 1; k <= col; ++k) sum = sum + SY(k, i) * X1(p, col + k) / SY(i, i);
    X1(p, i) = X1(p, i) + sum;
  }
}

/* heap of the breakpoints t[1..n] (iheap == 0: build it first); the least moves to t[n] */
static void hpsolb(int n, double *t, int *iorder, int iheap) {
  int    i, j, indxin, indxou;
  double ddum, out;
  if (iheap == 0) {
    for (int k = 2; k <= n; ++k) {
      ddum = X1(t, k);
      indxin = X1(iorder, k);
      i = k;
      while (i > 1) {
        j = i / 2;
        if (ddum < X1(t, j)) {
          X1(t, i) = X1(t, j);
          X1(iorder, i) = X1(iorder, j);
          i = j;
        } else {
          break;
        }
      }
      X1(t, i) = ddum;
      X1(iorder, i) = indxin;
    }
  }
  if (n > 1) {
    i = 1;
    out = X1(t, 1);
    indxou = X1(iorder, 1);
    ddum = X1(t, n);
    indxin = X1(iorder, n);
    for (;;) {
      j = i + i;
      if (j <= n - 1) {
        if (X1(t, j + 1) < X1(t, j)) j = j + 1;
        if (X1(t, j) < ddum) {
          X1(t, i) = X1(t, j);
          X1(iorder, i) = X1(iorder, j);
          i = j;
          continue;
        }
      }
      break;
    }
    X1(t, i) = ddum;
    X1(iorder, i) = indxin;
    X1(t, n) = out;
    X1(iorder, n) = indxou;
  }
}

/* the generalised Cauchy point xcp along the projected steepest descent path;
 * on return c = W'(xcp - x) (used by cmprlb) */
static void cauchy(int n, const double *x, const double *l, const double *u, const int *nbd, const double *g,
                   int *iorder, int *iwhere, double *t, double *d, double *xcp, int m, const double *wy,
                   const double *ws, const double *sy, const double *wt, double theta, int col, int head, double *p,
                   double *c, double *wbp, double *v, int *nseg, double sbgnrm, int *info, double epsmch) {
  int    bnded, xlower, xupper, nfree, nbreak, ibkmin, col2, pointr, nleft, ibp, iter;
  double bkmin, f1, f2, f2_org, dtm, tsum, tj, tj0, dt, dibp, zibp, dibp2, wmc, wmp, wmw, neggi, tl = 0.0, tu = 0.0;

  if (sbgnrm <= 0.0) {
    dcopy(n, x, xcp);
    return;
  }
  bnded = 1;
  nfree = n + 1;
  nbreak = 0;
  ibkmin = 0;
  bkmin = 0.0;
  col2 = 2 * col;
  f1 = 0.0;
  for (int i = 1; i <= col2; ++i) X1(p, i) = 0.0;

  for (int i = 1; i <= n; ++i) {
    neggi = -X1(g, i);
    if (X1(iwhere, i) != 3 && X1(iwhere, i) != -1) {
      if (X1(nbd, i) <= 2) tl = X1(x, i) - X1(l, i);
      if (X1(nbd, i) >= 2) tu = X1(u, i) - X1(x, i);
      xlower = X1(nbd, i) <= 2 && tl <= 0.0;
      xupper = X1(nbd, i) >= 2 && tu <= 0.0;
      X1(iwhere, i) = 0;
      if (xlower) {
        if (neggi <= 0.0) X1(iwhere, i) = 1;
      } else if (xupper) {
        if (neggi >= 0.0) X1(iwhere, i) = 2;
      } else {
        if (fabs(neggi) <= 0.0) X1(iwhere, i) = -3;
      }
    }
    pointr = head;
    if (X1(iwhere, i) != 0 && X1(iwhere, i) != -1) {
      X1(d, i) = 0.0;
    } else {
      X1(d, i) = neggi;
      f1 = f1 - neggi * neggi;
      for (int j = 1; j <= col; ++j) {
        X1(p, j) = X1(p, j) + WY(i, pointr) * neggi;
        X1(p, col + j) = X1(p, col + j) + WS(i, pointr) * neggi;
        pointr = pointr % m + 1;
      }
      if (X1(nbd, i) <= 2 && X1(nbd, i) != 0 && neggi < 0.0) {
        nbreak = nbreak + 1;
        X1(iorder, nbreak) = i;
        X1(t, nbreak) = tl / (-neggi);
        if (nbreak == 1 || X1(t, nbreak) < bkmin) {
          bkmin = X1(t, nbreak);
          ibkmin = nbreak;
        }
      } else if (X1(nbd, i) >= 2 && neggi > 0.0) {
        nbreak = nbreak + 1;
        X1(iorder, nbreak) = i;
        X1(t, nbreak) = tu / neggi;
        if (nbreak == 1 || X1(t, nbreak) < bkmin) {
          bkmin = X1(t, nbreak);
          ibkmin = nbreak;
        }
      } else {
        nfree = nfree - 1;
        X1(iorder, nfree) = i;
        if (fabs(neggi) > 0.0) bnded = 0;
      }
    }
  }

  if (theta != 1.0) dscal(col, theta, &X1(p, col + 1));
  dcopy(n, x, xcp);
  if (nbreak == 0 && nfree == n + 1) return;
  for (int j = 1; j <= col2; ++j) X1(c, j) = 0.0;

  f2 = -theta * f1;
  f2_org = f2;
  if (col > 0) {
    bmv(m, sy, wt, col, p, v, info);
    if (*info != 0) return;
    f2 = f2 - ddot(col2, v, p);
  }
  dtm = -f1 / f2;
  tsum = 0.0;
  *nseg = 1;
  if (nbreak == 0) goto locate;
  nleft = nbreak;
  iter = 1;
  tj = 0.0;

  for (;;) {
    tj0 = tj;
    if (iter == 1) {
      tj = bkmin;
      ibp = X1(iorder, ibkmin);
    } else {
      if (iter == 2) {
        if (ibkmin != nbreak) {
          X1(t, ibkmin) = X1(t, nbreak);
          X1(iorder, ibkmin) = X1(iorder, nbreak);
        }
      }
      hpsolb(nleft, t, iorder, iter - 2);
      tj = X1(t, nleft);
      ibp = X1(iorder, nleft);
    }
    dt = tj - tj0;
    if (dtm < dt) goto locate;

    tsum = tsum + dt;
    nleft = nleft - 1;
    iter = iter + 1;
    dibp = X1(d, ibp);
    X1(d, ibp) = 0.0;
    if (dibp > 0.0) {
      zibp = X1(u, ibp) - X1(x, ibp);
      X1(xcp, ibp) = X1(u, ibp);
      X1(iwhere, ibp) = 2;
    } else {
      zibp = X1(l, ibp) - X1(x, ibp);
      X1(xcp, ibp) = X1(l, ibp);
      X1(iwhere, ibp) = 1;
    }
    if (nleft == 0 && nbreak == n) {
      dtm = dt;
      goto update_c;
    }
    *nseg = *nseg + 1;
    dibp2 = dibp * dibp;
    f1 = f1 + dt * f2 + dibp2 - theta * dibp * zibp;
    f2 = f2 - theta * dibp2;
    if (col > 0) {
      daxpy(col2, dt, p, c);
      pointr = head;
      for (int j = 1; j <= col; ++j) {
        X1(wbp, j) = WY(ibp, pointr);
        X1(wbp, col + j) = theta * WS(ibp, pointr);
        pointr = pointr % m + 1;
      }
      bmv(m, sy, wt, col, wbp, v, info);
      if (*info != 0) return;
      wmc = ddot(col2, c, v);
      wmp = ddot(col2, p, v);
      wmw = ddot(col2, wbp, v);
      daxpy(col2, -dibp, wbp, p);
      f1 = f1 + dibp * wmc;
      f2 = f2 + 2.0 * dibp * wmp - dibp2 * wmw;
    }
    f2 = fmax(epsmch * f2_org, f2);
    if (nleft > 0) {
      dtm = -f1 / f2;
      continue;
    } else if (bnded) {
      f1 = 0.0;
      f2 = 0.0;
      dtm = 0.0;
    } else {
      dtm = -f1 / f2;
    }
    break;
  }

locate:
  if (dtm <= 0.0) dtm = 0.0;
  tsum = tsum + dtm;
  daxpy(n, tsum, d, xcp);
update_c:
  if (col > 0) daxpy(col2, dtm, p, c);
}

/* the entering / leaving variables and the free (index[1..nfree]) and active sets at the GCP */
static void freev(int n, int *nfree, int *index, int *nenter, int *ileave, int *indx2, const int *iwhere, int *wrk,
                  int updatd, int cnstnd, int iter) {
  *nenter = 0;
  *ileave = n + 1;
  if (iter > 0 && cnstnd) {
    for (int i = 1; i <= *nfree; ++i) {
      int k = X1(index, i);
      if (X1(iwhere, k) > 0) {
        *ileave = *ileave - 1;
        X1(indx2, *ileave) = k;
      }
    }
    for (int i = 1 + *nfree; i <= n; ++i) {
      int k = X1(index, i);
      if (X1(iwhere, k) <= 0) {
        *nenter = *nenter + 1;
        X1(indx2, *nenter) = k;
      }
    }
  }
  *wrk = (*ileave < n + 1) || (*nenter > 0) || updatd;
  *nfree = 0;
  int iact = n + 1;
  for (int i = 1; i <= n; ++i) {
    if (X1(iwhere, i) <= 0) {
      *nfree = *nfree + 1;
      X1(index, *nfree) = i;
    } else {
      iact = iact - 1;
      X1(index, iact) = i;
    }
  }
}

/* the LEL' factorisation of the indefinite matrix K of the subspace problem, in wn
 * (wn1 keeps the inner products of the previous iteration) */
static void formk(int n, int nsub, const int *ind, int nenter, int ileave, const int *indx2, int iupdat, int updatd,
                  double *wn, double *wn1, int m, const double *ws, const double *wy, const double *sy, double theta,
                  int col, int head, int *info) {
  int    ipntr, jpntr, iy, is, jy, js, is1, js1, k1, pbegin, pend, dbegin, dend, upcl, col2, m2;
  double temp1, temp2, temp3, temp4;

  if (updatd) {
    if (iupdat > m) {
      for (jy = 1; jy <= m - 1; ++jy) {
        js = m + jy;
        dcopy(m - jy, &WN1(jy + 1, jy + 1), &WN1(jy, jy));
        dcopy(m - jy, &WN1(js + 1, js + 1), &WN1(js, js));
        dcopy(m - 1, &WN1(m + 2, jy + 1), &WN1(m + 1, jy));
      }
    }
    pbegin = 1;
    pend = nsub;
    dbegin = nsub + 1;
    dend = n;
    iy = col;
    is = m + col;
    ipntr = head + col - 1;
    if (ipntr > m) ipntr = ipntr - m;
    jpntr = head;
    for (jy = 1; jy <= col; ++jy) {
      js = m + jy;
      temp1 = 0.0;
      temp2 = 0.0;
      temp3 = 0.0;
      for (int k = pbegin; k <= pend; ++k) {
        k1 = X1(ind, k);
        temp1 = temp1 + WY(k1, ipntr) * WY(k1, jpntr);
      }
      for (int k = dbegin; k <= dend; ++k) {
        k1 = X1(ind, k);
        temp2 = temp2 + WS(k1, ipntr) * WS(k1, jpntr);
        temp3 = temp3 + WS(k1, ipntr) * WY(k1, jpntr);
      }
      WN1(iy, jy) = temp1;
      WN1(is, js) = temp2;
      WN1(is, jy) = temp3;
      jpntr = jpntr % m + 1;
    }
    jy = col;
    jpntr = head + col - 1;
    if (jpntr > m) jpntr = jpntr - m;
    ipntr = head;
    for (int i = 1; i <= col; ++i) {
      is = m + i;
      temp3 = 0.0;
      for (int k = pbegin; k <= pend; ++k) {
        k1 = X1(ind, k);
        temp3 = temp3 + WS(k1, ipntr) * WY(k1, jpntr);
      }
      ipntr = ipntr % m + 1;
      WN1(is, jy) = temp3;
    }
    upcl = col - 1;
  } else {
    upcl = col;
  }

  ipntr = head;
  for (iy = 1; iy <= upcl; ++iy) {
    is = m + iy;
    jpntr = head;
    for (jy = 1; jy <= iy; ++jy) {
      js = m + jy;
      temp1 = 0.0;
      temp2 = 0.0;
      temp3 = 0.0;
      temp4 = 0.0;
      for (int k = 1; k <= nenter; ++k) {
        k1 = X1(indx2, k);
        temp1 = temp1 + WY(k1, ipntr) * WY(k1, jpntr);
        temp2 = temp2 + WS(k1, ipntr) * WS(k1, jpntr);
      }
      for (int k = ileave; k <= n; ++k) {
        k1 = X1(indx2, k);
        temp3 = temp3 + WY(k1, ipntr) * WY(k1, jpntr);
        temp4 = temp4 + WS(k1, ipntr) * WS(k1, jpntr);
      }
      WN1(iy, jy) = WN1(iy, jy) + temp1 - temp3;
      WN1(is, js) = WN1(is, js) - temp2 + temp4;
      jpntr = jpntr % m + 1;
    }
    ipntr = ipntr % m + 1;
  }

  ipntr = head;
  for (is = m + 1; is <= m + upcl; ++is) {
    jpntr = head;
    for (jy = 1; jy <= upcl; ++jy) {
      temp1 = 0.0;
      temp3 = 0.0;
      for (int k = 1; k <= nenter; ++k) {
        k1 = X1(indx2, k);
        temp1 = temp1 + WS(k1, ipntr) * WY(k1, jpntr);
      }
      for (int k = ileave; k <= n; ++k) {
        k1 = X1(indx2, k);
        temp3 = temp3 + WS(k1, ipntr) * WY(k1, jpntr);
      }
      if (is <= jy + m)
        WN1(is, jy) = WN1(is, jy) + temp1 - temp3;
      else
        WN1(is, jy) = WN1(is, jy) - temp1 + temp3;
      jpntr = jpntr % m + 1;
    }
    ipntr = ipntr % m + 1;
  }

  m2 = 2 * m;
  for (iy = 1; iy <= col; ++iy) {
    is = col + iy;
    is1 = m + iy;
    for (jy = 1; jy <= iy; ++jy) {
      js = col + jy;
      js1 = m + jy;
      WN(jy, iy) = WN1(iy, jy) / theta;
      WN(js, is) = WN1(is1, js1) * theta;
    }
    for (jy = 1; jy <= iy - 1; ++jy) WN(jy, is) = -WN1(is1, jy);
    for (jy = iy; jy <= col; ++jy) WN(jy, is) = WN1(is1, jy);
    WN(iy, iy) = WN(iy, iy) + SY(iy, iy);
  }

  dpofa(wn, m2, col, info);
  if (*info != 0) {
    *info = -1;
    return;
  }
  col2 = 2 * col;
  for (js = col + 1; js <= col2; ++js) dtrsl(wn, m2, col, &WN(1, js), 11, info);
  for (is = col + 1; is <= col2; ++is)
    for (js = is; js <= col2; ++js) WN(is, js) = WN(is, js) + ddot(col, &WN(1, is), &WN(1, js));
  dpofa(&WN(col + 1, col + 1), m2, col, info);
  if (*info != 0) {
    *info = -2;
    return;
  }
}

/* T = theta SS + L D^-1 L' in the upper triangle of wt, then its Cholesky factor J' */
static void formt(int m, double *wt, const double *sy, const double *ss, int col, double theta, int *info) {
  for (int j = 1; j <= col; ++j) WT(1, j) = theta * SS(1, j);
  for (int i = 2; i <= col; ++i) {
    for (int j = i; j <= col; ++j) {
      int    k1 = (i < j ? i : j) - 1;
      double ddum = 0.0;
      for (int k = 1; k <= k1; ++k) ddum = ddum + SY(i, k) * SY(j, k) / SY(k, k);
      WT(i, j) = ddum + theta * SS(i, j);
    }
  }
  dpofa(wt, m, col, info);
  if (*info != 0) *info = -3;
}

/* r = -Z'(B(xcp - x) + g), using wa[2m+1..4m] = W'(xcp - x) from cauchy */
static void cmprlb(int n, int m, const double *x, const double *g, const double *ws, const double *wy,
                   const double *sy, const double *wt, const double *z, double *r, double *wa, const int *index,
                   double theta, int col, int head, int nfree, int cnstnd, int *info) {
  if (!cnstnd && col > 0) {
    for (int i = 1; i <= n; ++i) X1(r, i) = -X1(g, i);
  } else {
    for (int i = 1; i <= nfree; ++i) {
      int k = X1(index, i);
      X1(r, i) = -theta * (X1(z, k) - X1(x, k)) - X1(g, k);
    }
    bmv(m, sy, wt, col, &X1(wa, 2 * m + 1), &X1(wa, 1), info);
    if (*info != 0) {
      *info = -8;
      return;
    }
    int pointr = head;
    for (int j = 1; j <= col; ++j) {
      double a1 = X1(wa, j), a2 = theta * X1(wa, col + j);
      for (int i = 1; i <= nfree; ++i) {
        int k = X1(index, i);
        X1(r, i) = X1(r, i) + WY(k, pointr) * a1 + WS(k, pointr) * a2;
      }
      pointr = pointr % m + 1;
    }
  }
}

/* the subspace minimisation over the free variables at the GCP, x (the GCP on entry) becomes
 * the subspace minimiser projected onto the box, or a step back towards the GCP when that
 * projection is not a descent direction from xx (version 3.0) */
static void subsm(int n, int m, int nsub, const int *ind, const double *l, const double *u, const int *nbd,
                  double *x, double *d, double *xp, const double *ws, const double *wy, double theta,
                  const double *xx, const double *gg, int col, int head, int *iword, double *wv, const double *wn,
                  int *info) {
  int    pointr, m2, col2, js, ibd, k;
  double temp1, temp2, alpha, dk, xk, dd_p;

  if (nsub <= 0) return;
  pointr = head;
  for (int i = 1; i <= col; ++i) {
    temp1 = 0.0;
    temp2 = 0.0;
    for (int j = 1; j <= nsub; ++j) {
      k = X1(ind, j);
      temp1 = temp1 + WY(k, pointr) * X1(d, j);
      temp2 = temp2 + WS(k, pointr) * X1(d, j);
    }
    X1(wv, i) = temp1;
    X1(wv, col + i) = theta * temp2;
    pointr = pointr % m + 1;
  }
  m2 = 2 * m;
  col2 = 2 * col;
  dtrsl(wn, m2, col2, wv, 11, info);
  if (*info != 0) return;
  for (int i = 1; i <= col; ++i) X1(wv, i) = -X1(wv, i);
  dtrsl(wn, m2, col2, wv, 1, info);
  if (*info != 0) return;
  pointr = head;
  for (int jy = 1; jy <= col; ++jy) {
    js = col + jy;
    for (int i = 1; i <= nsub; ++i) {
      k = X1(ind, i);
      X1(d, i) = X1(d, i) + WY(k, pointr) * X1(wv, jy) / theta + WS(k, pointr) * X1(wv, js);
    }
    pointr = pointr % m + 1;
  }
  dscal(nsub, 1.0 / theta, d);

  *iword = 0;
  dcopy(n, x, xp);
  for (int i = 1; i <= nsub; ++i) {
    k = X1(ind, i);
    dk = X1(d, i);
    xk = X1(x, k);
    if (X1(nbd, k) != 0) {
      if (X1(nbd, k) == 1) {
        X1(x, k) = fmax(X1(l, k), xk + dk);
        if (X1(x, k) == X1(l, k)) *iword = 1;
      } else if (X1(nbd, k) == 2) {
        xk = fmax(X1(l, k), xk + dk);
        X1(x, k) = fmin(X1(u, k), xk);
        if (X1(x, k) == X1(l, k) || X1(x, k) == X1(u, k)) *iword = 1;
      } else if (X1(nbd, k) == 3) {
        X1(x, k) = fmin(X1(u, k), xk + dk);
        if (X1(x, k) == X1(u, k)) *iword = 1;
      }
    } else {
      X1(x, k) = xk + dk;
    }
  }
  if (*iword == 0) return;

  dd_p = 0.0;
  for (int i = 1; i <= n; ++i) dd_p = dd_p + (X1(x, i) - X1(xx, i)) * X1(gg, i);
  if (dd_p > 0.0)
    dcopy(n, xp, x);
  else
    return;

  alpha = 1.0;
  temp1 = alpha;
  ibd = 0;
  for (int i = 1; i <= nsub; ++i) {
    k = X1(ind, i);
    dk = X1(d, i);
    if (X1(nbd, k) != 0) {
      if (dk < 0.0 && X1(nbd, k) <= 2) {
        temp2 = X1(l, k) - X1(x, k);
        if (temp2 >= 0.0)
          temp1 = 0.0;
        else if (dk * alpha < temp2)
          temp1 = temp2 / dk;
      } else if (dk > 0.0 && X1(nbd, k) >= 2) {
        temp2 = X1(u, k) - X1(x, k);
        if (temp2 <= 0.0)
          temp1 = 0.0;
        else if (dk * alpha > temp2)
          temp1 = temp2 / dk;
      }
      if (temp1 < alpha) {
        alpha = temp1;
        ibd = i;
      }
    }
  }
  if (alpha < 1.0) {
    dk = X1(d, ibd);
    k = X1(ind, ibd);
    if (dk > 0.0) {
      X1(x, k) = X1(u, k);
      X1(d, ibd) = 0.0;
    } else if (dk < 0.0) {
      X1(x, k) = X1(l, k);
      X1(d, ibd) = 0.0;
    }
  }
  for (int i = 1; i <= nsub; ++i) {
    k = X1(ind, i);
    X1(x, k) = X1(x, k) + alpha * X1(d, i);
  }
  *iword = alpha < 1.0 ? 1 : 0;
}

/* one step of the line search along d from t = x_k (r = g_k keeps the gradient there) */
static void lnsrlb(int n, const double *l, const double *u, const int *nbd, double *x, double f, double *fold,
                   double *gd, double *gdold, const double *g, const double *d, double *r, double *t, const double *z,
                   double *stp, double *dnorm, double *dtd, double *xstep, double *stpmx, int iter, int *ifun,
                   int *iback, int *nfgv, int *info, int *task, int boxed, int cnstnd, int *csave, int *isave,
                   double *dsave) {
  const double big = 1e10, ftol = 1e-3, gtol = 0.9, xtol = 0.1;

  if (*task != FG_LN) {
    *dtd = ddot(n, d, d);
    *dnorm = sqrt(*dtd);
    *stpmx = big;
    if (cnstnd) {
      if (iter == 0) {
        *stpmx = 1.0;
      } else {
        for (int i = 1; i <= n; ++i) {
          double a1 = X1(d, i);
          if (X1(nbd, i) != 0) {
            if (a1 < 0.0 && X1(nbd, i) <= 2) {
              double a2 = X1(l, i) - X1(x, i);
              if (a2 >= 0.0)
                *stpmx = 0.0;
              else if (a1 * *stpmx < a2)
                *stpmx = a2 / a1;
            } else if (a1 > 0.0 && X1(nbd, i) >= 2) {
              double a2 = X1(u, i) - X1(x, i);
              if (a2 <= 0.0)
                *stpmx = 0.0;
              else if (a1 * *stpmx > a2)
                *stpmx = a2 / a1;
            }
          }
        }
      }
    }
    if (iter == 0 && !boxed)
      *stp = fmin(1.0 / *dnorm, *stpmx);
    else
      *stp = 1.0;
    dcopy(n, x, t);
    dcopy(n, g, r);
    *fold = f;
    *ifun = 0;
    *iback = 0;
    *csave = LS_START;
  }
  *gd = ddot(n, g, d);
  if (*ifun == 0) {
    *gdold = *gd;
    if (*gd >= 0.0) {  /* not a descent direction: no line search is possible */
      *info = -4;
      return;
    }
  }
  dcsrch(f, *gd, stp, ftol, gtol, xtol, 0.0, *stpmx, csave, isave, dsave);
  *xstep = *stp * *dnorm;
  if (*csave != LS_CONV && !(*csave >= LS_WARN && *csave < LS_ERROR)) {
    *task = FG_LN;
    *ifun = *ifun + 1;
    *nfgv = *nfgv + 1;
    *iback = *ifun - 1;
    if (*stp == 1.0) {
      dcopy(n, z, x);
    } else {
      for (int i = 1; i <= n; ++i) X1(x, i) = *stp * X1(d, i) + X1(t, i);
    }
  } else {
    *task = NEW_X;
  }
}

/* append the newest correction pair (s, y) = (d, r) to WS / WY and update SS, SY, theta */
static void matupd(int n, int m, double *ws, double *wy, double *sy, double *ss, const double *d, const double *r,
                   int *itail, int iupdat, int *col, int *head, double *theta, double rr, double dr, double stp,
                   double dtd) {
  if (iupdat <= m) {
    *col = iupdat;
    *itail = (*head + iupdat - 2) % m + 1;
  } else {
    *itail = *itail % m + 1;
    *head = *head % m + 1;
  }
  dcopy(n, d, &WS(1, *itail));
  dcopy(n, r, &WY(1, *itail));
  *theta = rr / dr;
  if (iupdat > m) {
    for (int j = 1; j <= *col - 1; ++j) {
      dcopy(j, &SS(2, j + 1), &SS(1, j));
      dcopy(*col - j, &SY(j + 1, j + 1), &SY(j, j));
    }
  }
  int pointr = *head;
  for (int j = 1; j <= *col - 1; ++j) {
    SY(*col, j) = ddot(n, d, &WY(1, pointr));
    SS(j, *col) = ddot(n, &WS(1, pointr), d);
    pointr = pointr % m + 1;
  }
  if (stp == 1.0)
    SS(*col, *col) = dtd;
  else
    SS(*col, *col) = stp * stp * dtd;
  SY(*col, *col) = dr;
}

/* the infinity norm of the projected gradient */
static double projgr(int n, const double *l, const double *u, const int *nbd, const double *x, const double *g) {
  double sbgnrm = 0.0;
  for (int i = 1; i <= n; ++i) {
    double gi = X1(g, i);
    if (X1(nbd, i) != 0) {
      if (gi < 0.0) {
        if (X1(nbd, i) >= 2) gi = fmax(X1(x, i) - X1(u, i), gi);
      } else {
        if (X1(nbd, i) <= 2) gi = fmin(X1(x, i) - X1(l, i), gi);
      }
    }
    sbgnrm = fmax(sbgnrm, fabs(gi));
  }
  return sbgnrm;
}

static void errclb(int n, int m, double factr, const double *l, const double *u, const int *nbd, int *task,
                   int *info, int *k) {
  if (n <= 0) *task = ERROR_N0;
  if (m <= 0) *task = ERROR_M0;
  if (factr < 0.0) *task = ERROR_FACTR;
  for (int i = 1; i <= n; ++i) {
    if (X1(nbd, i) < 0 || X1(nbd, i) > 3) {
      *task = ERROR_NBD;
      *info = -6;
      *k = i;
    }
    if (X1(nbd, i) == 2 && X1(l, i) > X1(u, i)) {
      *task = ERROR_FEAS;
      *info = -7;
      *k = i;
    }
  }
}

/* ---------------------------------------------------------------------------------------------
 * mainlb: the iteration, suspended at every request for f and g (FG_ST, FG_LN) and at every
 * new iterate (NEW_X).  Its scalars live in isave[0..22] / dsave[0..15] between calls; the line
 * search keeps its own in isave[42..43] / dsave[16..28].
 * ------------------------------------------------------------------------------------------- */
enum { I_NINTOL, I_ITFILE, I_IBACK, I_NSKIP, I_HEAD, I_COL, I_ITAIL, I_ITER, I_IUPDAT, I_NSEG, I_NFGV, I_INFO,
       I_IFUN, I_IWORD, I_NFREE, I_NACT, I_ILEAVE, I_NENTER, I_LS = 42 };
enum { D_THETA, D_FOLD, D_TOL, D_DNORM, D_EPSMCH, D_GD, D_STPMX, D_SBGNRM, D_STP, D_GDOLD, D_DTD, D_LS = 16 };

static void mainlb(int n, int m, double *x, const double *l, const double *u, const int *nbd, double *f, double *g,
                   double factr, double pgtol, double *ws, double *wy, double *sy, double *ss, double *wt,
                   double *wn, double *snd, double *z, double *r, double *d, double *t, double *xp, double *wa,
                   int *index, int *iwhere, int *indx2, int *task, int *csave, int *lsave, int *isave,
                   double *dsave) {
  int    prjctd, cnstnd, boxed, updatd, wrk = 0;
  int    nintol, itfile, iback, nskip, head, col, itail, iter, iupdat, nseg, nfgv, info, ifun, iword, nfree, nact,
         ileave, nenter, k = 0;
  double theta, fold, tol, dnorm, epsmch, gd, stpmx, sbgnrm, stp, gdold, dtd, xstep, ddum, rr, dr;

  if (*task == START) {
    epsmch = DBL_EPSILON;
    col = 0;
    head = 1;
    theta = 1.0;
    iupdat = 0;
    updatd = 0;
    iback = 0;
    itail = 0;
    iword = 0;
    nact = 0;
    ileave = 0;
    nenter = 0;
    fold = 0.0;
    dnorm = 0.0;
    gd = 0.0;
    stpmx = 0.0;
    sbgnrm = 0.0;
    stp = 0.0;
    gdold = 0.0;
    dtd = 0.0;
    iter = 0;
    nfgv = 0;
    nseg = 0;
    nintol = 0;
    nskip = 0;
    nfree = n;
    ifun = 0;
    tol = factr * epsmch;
    info = 0;
    itfile = 0;
    errclb(n, m, factr, l, u, nbd, task, &info, &k);
    if (IS_ERROR(*task)) {
      prjctd = cnstnd = boxed = 0;
      goto save;
    }
    active(n, l, u, nbd, x, iwhere, &prjctd, &cnstnd, &boxed);
  } else {
    prjctd = lsave[0];
    cnstnd = lsave[1];
    boxed = lsave[2];
    updatd = lsave[3];
    nintol = isave[I_NINTOL];
    itfile = isave[I_ITFILE];
    iback = isave[I_IBACK];
    nskip = isave[I_NSKIP];
    head = isave[I_HEAD];
    col = isave[I_COL];
    itail = isave[I_ITAIL];
    iter = isave[I_ITER];
    iupdat = isave[I_IUPDAT];
    nseg = isave[I_NSEG];
    nfgv = isave[I_NFGV];
    info = isave[I_INFO];
    ifun = isave[I_IFUN];
    iword = isave[I_IWORD];
    nfree = isave[I_NFREE];
    nact = isave[I_NACT];
    ileave = isave[I_ILEAVE];
    nenter = isave[I_NENTER];
    theta = dsave[D_THETA];
    fold = dsave[D_FOLD];
    tol = dsave[D_TOL];
    dnorm = dsave[D_DNORM];
    epsmch = dsave[D_EPSMCH];
    gd = dsave[D_GD];
    stpmx = dsave[D_STPMX];
    sbgnrm = dsave[D_SBGNRM];
    stp = dsave[D_STP];
    gdold = dsave[D_GDOLD];
    dtd = dsave[D_DTD];

    if (*task == FG_LN) goto line_search;
    if (*task == NEW_X) goto new_x;
    if (*task == FG_ST) goto first_fg;
    if (IS_STOP(*task)) {
      if (*task == STOP_CPU) {
        dcopy(n, t, x);
        dcopy(n, r, g);
        *f = fold;
      }
      goto save;
    }
  }

  *task = FG_ST;
  goto save;

first_fg:
  nfgv = 1;
  sbgnrm = projgr(n, l, u, nbd, x, g);
  if (sbgnrm <= pgtol) {
    *task = CONV_GRAD;
    goto save;
  }

  for (;;) { /* one iteration */
    iword = -1;
    if (!cnstnd && col > 0) {
      dcopy(n, x, z);
      wrk = updatd;
      nseg = 0;
    } else {
      cauchy(n, x, l, u, nbd, g, indx2, iwhere, t, d, z, m, wy, ws, sy, wt, theta, col, head, &X1(wa, 1),
             &X1(wa, 2 * m + 1), &X1(wa, 4 * m + 1), &X1(wa, 6 * m + 1), &nseg, sbgnrm, &info, epsmch);
      if (info != 0) { /* singular triangular system: refresh the memory */
        info = 0;
        col = 0;
        head = 1;
        theta = 1.0;
        iupdat = 0;
        updatd = 0;
        continue;
      }
      nintol = nintol + nseg;
      freev(n, &nfree, index, &nenter, &ileave, indx2, iwhere, &wrk, updatd, cnstnd, iter);
      nact = n - nfree;
    }

    if (nfree != 0 && col != 0) {
      if (wrk) formk(n, nfree, index, nenter, ileave, indx2, iupdat, updatd, wn, snd, m, ws, wy, sy, theta, col, head,
                     &info);
      if (info != 0) { /* K not positive definite: refresh the memory */
        info = 0;
        col = 0;
        head = 1;
        theta = 1.0;
        iupdat = 0;
        updatd = 0;
        continue;
      }
      cmprlb(n, m, x, g, ws, wy, sy, wt, z, r, wa, index, theta, col, head, nfree, cnstnd, &info);
      if (info == 0)
        subsm(n, m, nfree, index, l, u, nbd, z, r, xp, ws, wy, theta, x, g, col, head, &iword, wa, wn, &info);
      if (info != 0) { /* singular triangular system: refresh the memory */
        info = 0;
        col = 0;
        head = 1;
        theta = 1.0;
        iupdat = 0;
        updatd = 0;
        continue;
      }
    }

    for (int i = 1; i <= n; ++i) X1(d, i) = X1(z, i) - X1(x, i);

  line_search:
    lnsrlb(n, l, u, nbd, x, *f, &fold, &gd, &gdold, g, d, r, t, z, &stp, &dnorm, &dtd, &xstep, &stpmx, iter, &ifun,
           &iback, &nfgv, &info, task, boxed, cnstnd, csave, &isave[I_LS], &dsave[D_LS]);
    if (info != 0 || iback >= 20) {
      dcopy(n, t, x); /* back to the previous iterate */
      dcopy(n, r, g);
      *f = fold;
      if (col == 0) {
        if (info == 0) {
          info = -9;
          nfgv = nfgv - 1;
          ifun = ifun - 1;
          iback = iback - 1;
        }
        *task = ABNORMAL;
        iter = iter + 1;
        goto save;
      }
      if (info == 0) nfgv = nfgv - 1;
      info = 0;
      col = 0;
      head = 1;
      theta = 1.0;
      iupdat = 0;
      updatd = 0;
      *task = RESTART;
      continue;
    } else if (*task == FG_LN) {
      goto save;
    }
    iter = iter + 1;
    sbgnrm = projgr(n, l, u, nbd, x, g);
    goto save; /* task == NEW_X */

  new_x:
    if (sbgnrm <= pgtol) {
      *task = CONV_GRAD;
      goto save;
    }
    ddum = fmax(fmax(fabs(fold), fabs(*f)), 1.0);
    if ((fold - *f) <= tol * ddum) {
      *task = CONV_F;
      if (iback >= 10) info = -5;
      goto save;
    }
    for (int i = 1; i <= n; ++i) X1(r, i) = X1(g, i) - X1(r, i);
    rr = ddot(n, r, r);
    if (stp == 1.0) {
      dr = gd - gdold;
      ddum = -gdold;
    } else {
      dr = (gd - gdold) * stp;
      dscal(n, stp, d);
      ddum = -gdold * stp;
    }
    if (dr <= epsmch * ddum) { /* skip the update */
      nskip = nskip + 1;
      updatd = 0;
      continue;
    }
    updatd = 1;
    iupdat = iupdat + 1;
    matupd(n, m, ws, wy, sy, ss, d, r, &itail, iupdat, &col, &head, &theta, rr, dr, stp, dtd);
    formt(m, wt, sy, ss, col, theta, &info);
    if (info != 0) { /* T not positive definite: refresh the memory */
      info = 0;
      col = 0;
      head = 1;
      theta = 1.0;
      iupdat = 0;
      updatd = 0;
    }
  }

save:
  lsave[0] = prjctd;
  lsave[1] = cnstnd;
  lsave[2] = boxed;
  lsave[3] = updatd;
  isave[I_NINTOL] = nintol;
  isave[I_ITFILE] = itfile;
  isave[I_IBACK] = iback;
  isave[I_NSKIP] = nskip;
  isave[I_HEAD] = head;
  isave[I_COL] = col;
  isave[I_ITAIL] = itail;
  isave[I_ITER] = iter;
  isave[I_IUPDAT] = iupdat;
  isave[I_NSEG] = nseg;
  isave[I_NFGV] = nfgv;
  isave[I_INFO] = info;
  isave[I_IFUN] = ifun;
  isave[I_IWORD] = iword;
  isave[I_NFREE] = nfree;
  isave[I_NACT] = nact;
  isave[I_ILEAVE] = ileave;
  isave[I_NENTER] = nenter;
  dsave[D_THETA] = theta;
  dsave[D_FOLD] = fold;
  dsave[D_TOL] = tol;
  dsave[D_DNORM] = dnorm;
  dsave[D_EPSMCH] = epsmch;
  dsave[D_GD] = gd;
  dsave[D_STPMX] = stpmx;
  dsave[D_SBGNRM] = sbgnrm;
  dsave[D_STP] = stp;
  dsave[D_GDOLD] = gdold;
  dsave[D_DTD] = dtd;
}

/* Minimises f over l <= x <= u (nbd[i]: 0 unbounded, 1 lower, 2 both, 3 upper bound) by reverse
 * communication: call with *task = START, then again after every return while the task is FG
 * (store f and g at x) or NEW_X (x is the next iterate); any other task ends the run. */
int setulb(int *n, int *m, double *x, double *l, double *u, int *nbd, double *f, double *g, double *factr,
           double *pgtol, double *wa, int *iwa, int *task, int *iprint, int *csave, int *lsave, int *isave,
           double *dsave) {
  (void)iprint;
  const int    nn = *n, mm = *m;
  const size_t lws = 0, lwy = lws + (size_t)mm * nn, lsy = lwy + (size_t)mm * nn, lss = lsy + (size_t)mm * mm,
               lwt = lss + (size_t)mm * mm, lwn = lwt + (size_t)mm * mm, lsnd = lwn + 4 * (size_t)mm * mm,
               lz = lsnd + 4 * (size_t)mm * mm, lr = lz + nn, ld = lr + nn, lt = ld + nn, lxp = lt + nn,
               lwa = lxp + nn;
  if (*task == START) {
    memset(isave, 0, 44 * sizeof(int));
    memset(dsave, 0, 29 * sizeof(double));
    memset(lsave, 0, 4 * sizeof(int));
  }
  mainlb(nn, mm, x, l, u, nbd, f, g, *factr, *pgtol, wa + lws, wa + lwy, wa + lsy, wa + lss, wa + lwt, wa + lwn,
         wa + lsnd, wa + lz, wa + lr, wa + ld, wa + lt, wa + lxp, wa + lwa, iwa, iwa + nn, iwa + 2 * nn, task, csave,
         lsave, isave, dsave);
  return 0;
}
