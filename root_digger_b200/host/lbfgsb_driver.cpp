// lbfgsb_driver.cpp -- binds L-BFGS-B 3.0 (setulb(), root_digger_b200/lbfgsb/lbfgsb.c,
// the interface of the C translation RootDigger vendors under lib/lbfgsb) at run time:
// lib/liblbfgsb.so is compiled by root_digger_b200/_build.py and loaded here from the
// directory of this library.  There is no substitute optimiser: if the library is
// missing, parameter optimisation fails loudly.
#include "lbfgsb_driver.hpp"

#include <dlfcn.h>

#include <mutex>
#include <stdexcept>
#include <string>

namespace rd {

static setulb_fn  g_setulb = nullptr;
static std::mutex g_mu;

setulb_fn load_setulb() {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_setulb) return g_setulb;
  std::string dir;
  Dl_info     info;
  if (dladdr((void *)&load_setulb, &info) && info.dli_fname) {
    dir = info.dli_fname;
    auto p = dir.rfind('/');
    dir = p == std::string::npos ? "." : dir.substr(0, p);
  }
  const char *env = getenv("RD_LBFGSB_LIB");
  std::string cands[] = {env ? env : "", dir + "/liblbfgsb.so", dir + "/../../root_digger_b200/lib/liblbfgsb.so",
                         "liblbfgsb.so"};
  void       *h = nullptr;
  for (auto &c : cands) {
    if (c.empty()) continue;
    h = dlopen(c.c_str(), RTLD_NOW | RTLD_LOCAL);
    if (h) break;
  }
  if (!h) throw std::runtime_error("liblbfgsb.so (L-BFGS-B 3.0) could not be loaded");
  g_setulb = (setulb_fn)dlsym(h, "setulb");
  if (!g_setulb) throw std::runtime_error("setulb not found in liblbfgsb.so");
  return g_setulb;
}

}  // namespace rd
