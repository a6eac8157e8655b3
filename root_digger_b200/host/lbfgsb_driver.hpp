#ifndef RD_HOST_LBFGSB_DRIVER_HPP_
#define RD_HOST_LBFGSB_DRIVER_HPP_
namespace rd {
// signature of setulb (root_digger_b200/lbfgsb/lbfgsb.c; RootDigger's lib/lbfgsb/lbfgsb.h, logical == int)
typedef int (*setulb_fn)(int *n, int *m, double *x, double *l, double *u, int *nbd, double *f, double *g,
                         double *factr, double *pgtol, double *wa, int *iwa, int *task, int *iprint,
                         int *csave, int *lsave, int *isave, double *dsave);
setulb_fn load_setulb();
// task codes of the C translation (lib/lbfgsb/lbfgsb.h:70-77)
enum { LBFGSB_START = 1, LBFGSB_NEW_X = 2, LBFGSB_FG = 10, LBFGSB_FG_END = 15 };
inline bool lbfgsb_is_fg(int task) { return task >= LBFGSB_FG && task <= LBFGSB_FG_END; }
}  // namespace rd
#endif
