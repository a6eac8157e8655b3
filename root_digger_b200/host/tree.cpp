// tree.cpp -- host-side traversal scheduler (see tree.hpp).
//
// Behavioural reference: RootDigger src/tree.cpp (root enumeration :174-189,
// virtual root insertion :213-236/:273-320, op schedule :364-441, root-move
// schedule :572-657, ranking :863-940, NHX/newick :443-492,:691-762) and the
// coraxlib utree conventions in SURVEY.md Appendix A-7 (index numbering pinned
// by the reference's known-answer tests test/src/tree.cpp:142-212,410-433).
#include "tree.hpp"

#include <algorithm>
#include <cctype>
#include <cstring>
#include <cmath>
#include <cstdlib>
#include <fstream>
#include <limits>
#include <numeric>
#include <sstream>

namespace rd {

// ---------------------------------------------------------------------------
// newick parsing
// ---------------------------------------------------------------------------
namespace {

struct pnode {
  std::vector<std::unique_ptr<pnode>> kids;
  std::string                         label;
  bool                                has_label = false;
  double                              length = 0.0;
};

class newick_reader {
public:
  explicit newick_reader(const std::string &s) : _s(s) {}

  std::unique_ptr<pnode> read_tree() {
    skip();
    auto root = read_subtree();
    skip();
    if (_i >= _s.size() || _s[_i] != ';') throw std::invalid_argument("newick: missing ';'");
    return root;
  }

private:
  void skip() {
    for (;;) {
      while (_i < _s.size() && std::isspace((unsigned char)_s[_i])) ++_i;
      if (_i < _s.size() && _s[_i] == '[') {  // comment
        while (_i < _s.size() && _s[_i] != ']') ++_i;
        if (_i < _s.size()) ++_i;
        continue;
      }
      break;
    }
  }

  std::unique_ptr<pnode> read_subtree() {
    auto n = std::make_unique<pnode>();
    skip();
    if (_i < _s.size() && _s[_i] == '(') {
      ++_i;
      for (;;) {
        n->kids.push_back(read_subtree());
        skip();
        if (_i >= _s.size()) throw std::invalid_argument("newick: unbalanced parentheses");
        if (_s[_i] == ',') {
          ++_i;
          continue;
        }
        if (_s[_i] == ')') {
          ++_i;
          break;
        }
        throw std::invalid_argument("newick: unexpected character");
      }
    }
    skip();
    // label
    if (_i < _s.size() && (_s[_i] == '\'' || _s[_i] == '"')) {
      char q = _s[_i++];
      while (_i < _s.size() && _s[_i] != q) n->label.push_back(_s[_i++]);
      if (_i < _s.size()) ++_i;
      n->has_label = true;
    } else {
      while (_i < _s.size() && !std::strchr("():,;[", _s[_i]) &&
             !std::isspace((unsigned char)_s[_i]))
        n->label.push_back(_s[_i++]);
      n->has_label = !n->label.empty();
    }
    skip();
    if (_i < _s.size() && _s[_i] == ':') {
      ++_i;
      skip();
      const char *b = _s.c_str() + _i;
      char       *e = nullptr;
      n->length = std::strtod(b, &e);
      if (e == b) throw std::invalid_argument("newick: bad branch length");
      _i += (size_t)(e - b);
    }
    if (n->kids.empty() && !n->has_label) throw std::invalid_argument("newick: unnamed tip");
    return n;
  }

  const std::string &_s;
  size_t             _i = 0;
};

unode_t *new_unode(utree_t &t) {
  t.arena.emplace_back();
  t.arena.back().uid = (unsigned int)t.arena.size() - 1;
  return &t.arena.back();
}

void join(unode_t *a, unode_t *b, double len) {
  a->back = b;
  b->back = a;
  a->length = b->length = len;
}

// returns the unode that faces the parent
unode_t *build(utree_t &t, const pnode &p) {
  unode_t *top = new_unode(t);
  top->label = p.label;
  top->has_label = p.has_label;
  top->length = p.length;
  if (p.kids.empty()) {
    t.tip_count++;
    return top;
  }
  if (p.kids.size() != 2)
    throw std::invalid_argument("newick: only strictly bifurcating inner nodes are supported");
  unode_t *l = new_unode(t), *r = new_unode(t);
  top->next = l;
  l->next = r;
  r->next = top;
  l->label = r->label = p.label;
  l->has_label = r->has_label = p.has_label;
  unode_t *cl = build(t, *p.kids[0]);
  unode_t *cr = build(t, *p.kids[1]);
  join(l, cl, cl->length);
  join(r, cr, cr->length);
  t.inner_count++;
  return top;
}

// index numbering of corax_utree_reset_template_indices: tips 0..n-1 and inner
// nodes n.. in post-order from vroot (vroot->back first); every edge carries
// the index of its child-side node as pmatrix index
struct counters {
  unsigned tip = 0, inner_clv = 0, inner_node = 0;
  int      scaler = 0;
};

void number_ring(unode_t *node, counters &c) {
  unode_t *s = node;
  do {
    s->clv_index = c.inner_clv;
    s->scaler_index = c.scaler;
    s->node_index = c.inner_node++;
    s = s->next;
  } while (s != node);
  c.inner_clv++;
  c.scaler++;
}

void number_subtree(unode_t *node, counters &c) {
  if (!node->next) {
    node->clv_index = node->pmatrix_index = node->node_index = c.tip++;
    node->scaler_index = RDK_SCALE_BUFFER_NONE;
    return;
  }
  for (unode_t *s = node->next; s != node; s = s->next) number_subtree(s->back, c);
  node->pmatrix_index = c.inner_clv;
  number_ring(node, c);
  for (unode_t *s = node->next; s != node; s = s->next) s->pmatrix_index = s->back->pmatrix_index;
}

void number_tree(utree_t &t) {
  counters c;
  c.inner_clv = c.inner_node = t.tip_count;
  unode_t *root = t.vroot;
  number_subtree(root->back, c);
  for (unode_t *s = root->next; s != root; s = s->next) number_subtree(s->back, c);
  number_ring(root, c);
  unode_t *s = root;
  do {
    s->pmatrix_index = s->back->pmatrix_index;
    s = s->next;
  } while (s != root);
  // the edge behind vroot->back is numbered by the node at its far end
  root->back->pmatrix_index = root->pmatrix_index;

  t.nodes.assign(t.tip_count + t.inner_count, nullptr);
  for (auto &u : t.arena) {
    if (!u.next)
      t.nodes[u.clv_index] = &u;
    else if (!t.nodes[u.clv_index])
      t.nodes[u.clv_index] = &u;
  }
  // represent every inner node by the unode that faces vroot's side (the first
  // one created), and vroot by itself
  t.nodes[root->clv_index] = root;
}

}  // namespace

std::unique_ptr<utree_t> utree_parse_newick_string_unroot(const std::string &newick) {
  newick_reader          rd(newick);
  std::unique_ptr<pnode> top = rd.read_tree();
  auto                   t = std::make_unique<utree_t>();
  if (top->kids.size() == 3) {
    unode_t *a = new_unode(*t), *b = new_unode(*t), *c = new_unode(*t);
    a->next = b;
    b->next = c;
    c->next = a;
    for (unode_t *u : {a, b, c}) {
      u->label = top->label;
      u->has_label = top->has_label;
    }
    unode_t *ring[3] = {a, b, c};
    for (int i = 0; i < 3; ++i) {
      unode_t *k = build(*t, *top->kids[i]);
      join(ring[i], k, k->length);
    }
    t->inner_count++;
    t->vroot = a;
  } else if (top->kids.size() == 2) {
    const pnode &l = *top->kids[0], &r = *top->kids[1];
    if (l.kids.empty() && r.kids.empty())
      throw std::invalid_argument("newick: a tree needs at least three tips");
    unode_t *lu = build(*t, l);
    unode_t *ru = build(*t, r);
    join(lu, ru, l.length + r.length);
    t->vroot = lu->next ? lu : ru;
  } else {
    throw std::invalid_argument("newick: the top level must have two or three children");
  }
  if (t->tip_count < 3) throw std::invalid_argument("newick: a tree needs at least three tips");
  t->edge_count = 2 * t->tip_count - 3;
  if (t->inner_count != t->tip_count - 2)
    throw std::invalid_argument("newick: tree is not strictly bifurcating");
  number_tree(*t);
  return t;
}

std::unique_ptr<utree_t> utree_parse_newick_unroot(const std::string &filename) {
  std::ifstream in(filename);
  if (!in) return nullptr;
  std::stringstream ss;
  ss << in.rdbuf();
  try {
    return utree_parse_newick_string_unroot(ss.str());
  } catch (const std::invalid_argument &) {
    return nullptr;
  }
}

std::unique_ptr<utree_t> utree_clone(const utree_t &src) {
  auto                                            t = std::make_unique<utree_t>();
  std::unordered_map<const unode_t *, unode_t *> m;
  for (const auto &u : src.arena) {
    t->arena.push_back(u);
    m[&u] = &t->arena.back();
  }
  for (auto &u : t->arena) {
    if (u.next) u.next = m.at(u.next);
    if (u.back) u.back = m.at(u.back);
  }
  t->tip_count = src.tip_count;
  t->inner_count = src.inner_count;
  t->edge_count = src.edge_count;
  t->nodes.reserve(src.nodes.size());
  for (auto *n : src.nodes) t->nodes.push_back(n ? m.at(n) : nullptr);
  t->vroot = m.at(src.vroot);
  return t;
}

namespace {
void traverse_rec(unode_t *node, const std::function<bool(unode_t *)> &accept,
                  std::vector<unode_t *> &out) {
  if (!accept(node)) return;
  if (node->next) {
    unode_t *s = node->next;
    do {
      traverse_rec(s->back, accept, out);
      s = s->next;
    } while (s && s != node);
  }
  out.push_back(node);
}
}  // namespace

std::vector<unode_t *> utree_traverse_postorder(unode_t *vroot,
                                                const std::function<bool(unode_t *)> &accept) {
  std::vector<unode_t *> out;
  if (!vroot->next) return out;
  traverse_rec(vroot->back, accept, out);
  traverse_rec(vroot, accept, out);
  return out;
}

void utree_create_operations(const std::vector<unode_t *> &trav, size_t count,
                             std::vector<double> &branches,
                             std::vector<unsigned int> &pmatrix_indices,
                             std::vector<rdk_operation_t> &ops) {
  branches.clear();
  pmatrix_indices.clear();
  ops.clear();
  for (size_t i = 0; i < count; ++i) {
    const unode_t *n = trav[i];
    // the far end of the last node's edge would duplicate that edge
    if (n != trav[count - 1]->back) {
      branches.push_back(n->length);
      pmatrix_indices.push_back(n->pmatrix_index);
    }
    if (n->next) {
      const unode_t  *a = n->next->back, *b = n->next->next->back;
      rdk_operation_t op;
      op.parent_clv_index = n->clv_index;
      op.parent_scaler_index = n->scaler_index;
      op.child1_clv_index = a->clv_index;
      op.child1_scaler_index = a->scaler_index;
      op.child1_matrix_index = a->pmatrix_index;
      op.child2_clv_index = b->clv_index;
      op.child2_scaler_index = b->scaler_index;
      op.child2_matrix_index = b->pmatrix_index;
      ops.push_back(op);
    }
  }
}

namespace {
std::string newick_rec(const unode_t *n, const std::function<std::string(const unode_t *)> &ser) {
  if (!n->next) return ser(n);
  std::string s = "(";
  bool        first = true;
  for (const unode_t *k = n->next; k != n; k = k->next) {
    if (!first) s += ",";
    s += newick_rec(k->back, ser);
    first = false;
  }
  s += ")";
  s += ser(n);
  return s;
}
}  // namespace

std::string utree_export_newick(const unode_t *vroot,
                                const std::function<std::string(const unode_t *)> &ser) {
  if (!vroot->next) vroot = vroot->back;
  std::string    s = "(";
  const unode_t *k = vroot;
  bool           first = true;
  do {
    if (!first) s += ",";
    s += newick_rec(k->back, ser);
    first = false;
    k = k->next;
  } while (k != vroot);
  s += ")";
  if (vroot->has_label) s += vroot->label;
  s += ";";
  return s;
}

}  // namespace rd

using rd::unode_t;

// ---------------------------------------------------------------------------
// rooted_tree_t
// ---------------------------------------------------------------------------
static void for_ring(unode_t *n, const std::function<void(unode_t *)> &f) {
  unode_t *s = n;
  do {
    f(s);
    s = s->next;
  } while (s != nullptr && s != n);
}
static void tag_nodes(unode_t *n) {
  for_ring(n, [](unode_t *u) { u->mark = 1; });
}
static void untag_nodes(unode_t *n) {
  for_ring(n, [](unode_t *u) { u->mark = 0; });
}

rooted_tree_t::rooted_tree_t(const std::string &tree_filename) {
  _tree = rd::utree_parse_newick_unroot(tree_filename);
  if (!_tree) throw std::invalid_argument("Tree file could not be parsed");
  init_from_tree();
}

rooted_tree_t rooted_tree_t::from_newick(const std::string &text) {
  rooted_tree_t t;
  t._tree = rd::utree_parse_newick_string_unroot(text);
  t.init_from_tree();
  return t;
}

void rooted_tree_t::init_from_tree() {
  _rooted = false;
  generate_root_locations();
  add_root_space();
  sort_root_locations();
}

rooted_tree_t::rooted_tree_t(rooted_tree_t &&o) noexcept
    : _tree(std::move(o._tree)), _root_left(o._root_left), _root_right(o._root_right),
      _current_rl(o._current_rl), _roots(std::move(o._roots)),
      _root_annotations(std::move(o._root_annotations)), _rooted(o._rooted) {
  o._root_left = o._root_right = nullptr;
}

rooted_tree_t &rooted_tree_t::operator=(rooted_tree_t &&o) noexcept {
  _tree = std::move(o._tree);
  _root_left = o._root_left;
  _root_right = o._root_right;
  _current_rl = o._current_rl;
  _roots = std::move(o._roots);
  _root_annotations = std::move(o._root_annotations);
  _rooted = o._rooted;
  o._root_left = o._root_right = nullptr;
  return *this;
}

rooted_tree_t::rooted_tree_t(const rooted_tree_t &other) { copy_from(other); }

rooted_tree_t &rooted_tree_t::operator=(const rooted_tree_t &other) {
  if (this != &other) copy_from(other);
  return *this;
}

// src/tree.cpp:26-37,131-164,764-802: a rooted tree may not be copied; root ids
// are carried over by position in the (identical) post-order traversal
void rooted_tree_t::copy_from(const rooted_tree_t &other) {
  if (other.rooted()) throw std::runtime_error{"Attempted to copy a tree that is rooted"};
  // clone only the unrooted part (the other tree's spare root unodes are
  // detached while it is unrooted)
  _tree = std::make_unique<rd::utree_t>();
  std::unordered_map<const unode_t *, unode_t *> m;
  for (const auto &u : other._tree->arena) {
    if (&u == other._root_left || &u == other._root_right) continue;
    _tree->arena.push_back(u);
    m[&u] = &_tree->arena.back();
  }
  for (auto &u : _tree->arena) {
    if (u.next) u.next = m.at(u.next);
    if (u.back) u.back = m.at(u.back);
    u.mark = 0;
    u.annotation.clear();
  }
  _tree->tip_count = other._tree->tip_count;
  _tree->inner_count = other._tree->inner_count;
  _tree->edge_count = other._tree->edge_count;
  for (size_t i = 0; i < (size_t)_tree->tip_count + _tree->inner_count; ++i)
    _tree->nodes.push_back(m.at(other._tree->nodes[i]));
  _tree->vroot = m.at(other._tree->vroot);
  _rooted = false;

  _roots.clear();
  std::unordered_map<const unode_t *, size_t> id_of;
  for (const auto &r : other.roots()) {
    id_of[r.edge] = r.id;
    id_of[r.edge->back] = r.id;
  }
  auto theirs = other.full_traverse();
  auto ours = full_traverse();
  if (theirs.size() != ours.size())
    throw std::runtime_error("Traversal sizes didn't match during copy "
                             "constructor, something is seriously wrong");
  std::unordered_set<size_t> used;
  for (size_t i = 0; i < theirs.size(); ++i) {
    auto it = id_of.find(theirs[i]);
    if (it != id_of.end() && !used.count(it->second)) {
      _roots.push_back({ours[i], it->second, ours[i]->length, 0.5});
      used.insert(it->second);
    }
  }
  if (_roots.size() != other._roots.size())
    throw std::runtime_error{"We got the wrong number of roots after copy"};
  sort_root_locations();

  _root_annotations.clear();
  for (const auto &kv : other._root_annotations) {
    auto it = m.find(kv.first);
    if (it != m.end()) _root_annotations[it->second] = kv.second;
  }
  add_root_space();
}

root_location_t rooted_tree_t::root_location(size_t index) const {
  if (index >= _roots.size())
    throw std::invalid_argument(std::string("Invalid index for roots on this tree: ") +
                                std::to_string(index));
  return _roots[index];
}

root_location_t rooted_tree_t::root_location(const std::string &name) const {
  for (const auto &rl : _roots)
    if (rl.edge->has_label && name == rl.edge->label) return rl;
  throw std::runtime_error{std::string{"Can't find the root location with label: "} + name};
}

std::unordered_map<std::string, unsigned int> rooted_tree_t::label_map() const {
  std::unordered_map<std::string, unsigned int> lm;
  if (!_tree) return lm;
  for (unsigned i = 0; i < tip_count(); ++i) lm[_tree->nodes[i]->label] = _tree->nodes[i]->clv_index;
  return lm;
}

std::unordered_set<std::string> rooted_tree_t::label_set() const {
  std::unordered_set<std::string> ls;
  if (!_tree) return ls;
  for (unsigned i = 0; i < tip_count(); ++i) ls.insert(_tree->nodes[i]->label);
  return ls;
}

void rooted_tree_t::sort_root_locations() {
  std::sort(_roots.begin(), _roots.end(),
            [](const root_location_t &a, const root_location_t &b) { return a.id < b.id; });
}

// src/tree.cpp:174-189: one root location per edge, id = position of the edge's
// first end point in the parse-time post-order
void rooted_tree_t::generate_root_locations() {
  auto                          edges = full_traverse();
  std::unordered_set<unode_t *> seen;
  _roots.clear();
  size_t id = 0;
  for (auto *e : edges) {
    if (!seen.count(e) && !seen.count(e->back)) {
      seen.insert(e);
      _roots.push_back({e, id++, e->length, 0.5});
    }
  }
}

std::vector<root_location_t> rooted_tree_t::internal_root_locations() const {
  std::vector<root_location_t> ret;
  for (const auto &rl : _roots)
    if (rl.is_internal()) ret.push_back(rl);
  return ret;
}

std::vector<root_location_t> rooted_tree_t::external_root_locations() const {
  std::vector<root_location_t> ret;
  for (const auto &rl : _roots)
    if (rl.is_external()) ret.push_back(rl);
  return ret;
}

// src/tree.cpp:213-236: two spare unodes that become the virtual root
void rooted_tree_t::add_root_space() {
  unsigned new_size = _tree->inner_count + _tree->tip_count + 1;
  unsigned total_unodes = _tree->inner_count * 3 + _tree->tip_count;
  _tree->arena.emplace_back();
  _root_left = &_tree->arena.back();
  _root_left->uid = (unsigned int)_tree->arena.size() - 1;
  _tree->arena.emplace_back();
  _root_right = &_tree->arena.back();
  _root_right->uid = (unsigned int)_tree->arena.size() - 1;
  _root_left->next = _root_right;
  _root_right->next = _root_left;
  _root_left->clv_index = _root_right->clv_index = new_size;
  _root_left->scaler_index = _root_right->scaler_index = (int)(_tree->inner_count - 1);
  _root_left->node_index = total_unodes + 1;
  _root_right->node_index = total_unodes + 2;
  _root_right->pmatrix_index = _tree->edge_count - 1;
  _tree->nodes.resize(new_size, nullptr);
  _tree->nodes[new_size - 1] = _root_left;
}

std::vector<unode_t *> rooted_tree_t::full_traverse() const {
  return rd::utree_traverse_postorder(_tree->vroot, [](unode_t *) { return true; });
}

// src/tree.cpp:273-320
void rooted_tree_t::root_by(const root_location_t &rl) {
  if (rl.edge == _tree->vroot) {
    update_root(rl);
    return;
  }
  if (rooted()) unroot();
  unsigned tree_size = _tree->inner_count + _tree->tip_count + 1;
  unode_t *rleft = _root_left, *rright = _root_right;
  rleft->next = rright;
  rright->next = rleft;

  unode_t *lchild = rl.edge;
  unode_t *rchild = lchild->back;

  lchild->back = rleft;
  rleft->back = lchild;
  lchild->length = rleft->length = rl.brlen();

  rchild->back = rright;
  rright->back = rchild;
  rchild->length = rright->length = rl.brlen_compliment();

  unsigned total_unodes = _tree->inner_count * 3 + _tree->tip_count;
  _tree->inner_count += 1;
  _tree->edge_count += 1;
  _tree->vroot = rleft;

  rleft->clv_index = rright->clv_index = tree_size - 1;
  rleft->scaler_index = rright->scaler_index = (int)(_tree->inner_count - 1);
  rleft->pmatrix_index = lchild->pmatrix_index;
  rright->node_index = total_unodes + 2;
  rchild->pmatrix_index = rright->pmatrix_index = _tree->edge_count - 1;

  _current_rl = rl;
  _rooted = true;
}

// src/tree.cpp:322-332
void rooted_tree_t::update_root(root_location_t root) {
  if (root.edge != _tree->vroot)
    throw std::runtime_error("Provided root doesn't match the current tree");
  unode_t *right_root = root.edge;
  unode_t *left_root = root.edge->next;
  right_root->length = right_root->back->length = root.brlen();
  left_root->length = left_root->back->length = root.brlen_compliment();
}

// src/tree.cpp:334-358
void rooted_tree_t::unroot() {
  unode_t *lchild = _tree->vroot->back;
  unode_t *rchild = _tree->vroot->next->back;
  unode_t *rleft = _tree->vroot, *rright = _tree->vroot->next;

  rchild->back = lchild;
  lchild->back = rchild;
  rchild->length = lchild->length = _current_rl.saved_brlen;

  for (unode_t *u : {rleft, rright}) {
    u->length = -1;
    u->node_index = std::numeric_limits<unsigned int>::max();
    u->back = nullptr;
  }
  _tree->vroot = lchild->next != nullptr ? lchild : rchild;
  if (_tree->vroot->next == nullptr) throw std::runtime_error("unrooted to a tip");
  _tree->inner_count -= 1;
  _tree->edge_count -= 1;
  rchild->pmatrix_index = lchild->pmatrix_index;
  _rooted = false;
}

bool rooted_tree_t::rooted() const { return _tree->vroot->next->next == _tree->vroot; }

static void fill_root_op(rdk_operation_t &op, const unode_t *root) {
  op.parent_clv_index = root->clv_index;
  op.parent_scaler_index = root->scaler_index;
  op.child1_clv_index = root->back->clv_index;
  op.child1_scaler_index = root->back->scaler_index;
  op.child1_matrix_index = root->back->pmatrix_index;
  op.child2_clv_index = root->next->back->clv_index;
  op.child2_scaler_index = root->next->back->scaler_index;
  op.child2_matrix_index = root->next->back->pmatrix_index;
}

// src/tree.cpp:364-413: full post-order schedule, n-2 inner ops + the root op,
// 2n-2 (pmatrix, branch length) pairs
rooted_tree_t::op_bundle_t rooted_tree_t::generate_operations(const root_location_t &new_root) {
  root_by(new_root);
  auto                         trav = full_traverse();
  std::vector<rdk_operation_t> ops;
  std::vector<unsigned int>    pm;
  std::vector<double>          br;
  rd::utree_create_operations(trav, trav.size() - 1, br, pm, ops);
  rdk_operation_t root_op;
  fill_root_op(root_op, trav.back());
  ops.push_back(root_op);
  return std::make_tuple(ops, pm, br);
}

// src/tree.cpp:415-441: the single root op and its two branches
std::tuple<rdk_operation_t, std::vector<unsigned int>, std::vector<double>>
rooted_tree_t::generate_derivative_operations(const root_location_t &root) {
  root_by(root);
  const unode_t  *v = _tree->vroot;
  rdk_operation_t op;
  fill_root_op(op, v);
  std::vector<unsigned int> pm{v->back->pmatrix_index, v->next->back->pmatrix_index};
  std::vector<double>       br{v->back->length, v->next->back->length};
  return std::make_tuple(op, pm, br);
}

// src/tree.cpp:538-570
void rooted_tree_t::find_path(unode_t *n1, unode_t *n2) {
  unode_t *start = n1, *cur = n1;
  do {
    if (find_path_recurse(cur->back, n2)) break;
    cur = cur->next;
  } while (cur != nullptr && cur != start);
}

bool rooted_tree_t::find_path_recurse(unode_t *n1, unode_t *n2) {
  if (n1 == n2) {
    tag_nodes(n1);
    return true;
  }
  if (!n1->next) return false;
  for (unode_t *s = n1->next; s != n1; s = s->next) {
    if (s == n2) {
      tag_nodes(s);
      return true;
    }
    if (find_path_recurse(s->back, n2)) {
      tag_nodes(s);
      return true;
    }
  }
  return false;
}

// src/tree.cpp:572-657: re-orient only the CLVs between the old and new root
rooted_tree_t::op_bundle_t
rooted_tree_t::generate_root_update_operations(const root_location_t &new_root) {
  // the reference dereferences the current root edge unconditionally (UB on a tree that
  // was never rooted); here that is an error the caller can see
  if (!rooted() || _current_rl.edge == nullptr)
    throw std::runtime_error("generate_root_update_operations: the tree has no current root "
                             "(call generate_operations / root_by first)");
  if (new_root.edge == _current_rl.edge || new_root.edge == _current_rl.edge->back) return {};

  auto old_root = _current_rl;
  root_by(new_root);
  find_path(old_root.edge, _tree->vroot);
  tag_nodes(old_root.edge);
  tag_nodes(old_root.edge->back);
  tag_nodes(_tree->vroot->back);
  tag_nodes(_tree->vroot->next->back);

  auto trav = rd::utree_traverse_postorder(_tree->vroot, [](unode_t *n) {
    if (n->mark) {
      n->mark = 0;
      return true;
    }
    return false;
  });
  if (trav.empty()) throw std::runtime_error("traversal buffer when updating the root had size zero");

  std::vector<rdk_operation_t> ops;
  std::vector<unsigned int>    pm;
  std::vector<double>          br;
  rd::utree_create_operations(trav, trav.size() - 1, br, pm, ops);
  rdk_operation_t root_op;
  fill_root_op(root_op, _tree->vroot);
  ops.push_back(root_op);

  clear_traversal_data();
  return std::make_tuple(ops, pm, br);
}

// ---- the directed-CLV placement sweep (see tree.hpp) --------------------------
namespace {
// height in edges of the subtree hanging below c (c faces up); diam = longest path seen
unsigned height_below(const unode_t *c, unsigned &diam) {
  if (!c->next) return 0;
  unsigned h1 = height_below(c->next->back, diam) + 1, h2 = height_below(c->next->next->back, diam) + 1;
  diam = std::max(diam, h1 + h2);
  return std::max(h1, h2);
}
}  // namespace

unsigned int rooted_tree_t::sweep_depth_bound() const {
  // the depth of any edge below any root edge is at most the diameter of the tree
  unsigned              diam = 0;
  std::vector<unsigned> tops;
  const unode_t        *v = _tree->vroot;
  const unode_t        *s = v;
  do {
    tops.push_back(height_below(s->back, diam) + 1);
    s = s->next;
  } while (s && s != v);
  std::sort(tops.rbegin(), tops.rend());
  if (tops.size() >= 2) diam = std::max(diam, tops[0] + tops[1]);
  return diam + 1;
}

rooted_tree_t::sweep_schedule_t rooted_tree_t::generate_sweep_operations(size_t begin, size_t end,
                                                                         unsigned int clv0, int scaler0,
                                                                         unsigned int pm0,
                                                                         unsigned int extra,
                                                                         const std::vector<double> &ratio) const {
  if (!rooted() || _current_rl.edge == nullptr)
    throw std::runtime_error("generate_sweep_operations: the tree has no current root "
                             "(call generate_operations / root_by first)");
  if (begin > end || end > _roots.size()) throw std::invalid_argument("generate_sweep_operations: bad root range");
  if (!ratio.empty() && ratio.size() != _roots.size())
    throw std::invalid_argument("generate_sweep_operations: one ratio per root location is needed");
  sweep_schedule_t out;
  if (begin == end) return out;
  {
    const size_t q = end - begin;  // one directed-CLV operation + one root operation per placement, at most
    out.ops.reserve(2 * q + 2);
    out.mi.reserve(4 * q + 4);
    out.bl.reserve(4 * q + 4);
    out.pm_off.reserve(q + 1);
    out.op_off.reserve(q + 1);
    out.root_pos.reserve(q);
  }

  const unode_t     *lchild = _tree->vroot->back, *rchild = _tree->vroot->next->back;
  const unsigned int ML = pm0, MR = pm0 + 1, MC = pm0 + 2;
  const double       L0 = _current_rl.saved_brlen;

  // position in roots() of the edge behind each unode (both end points), keyed by unode uid
  const size_t        n_unodes = _tree->arena.size();
  std::vector<size_t> pos_of(n_unodes, (size_t)-1);
  for (size_t i = 0; i < _roots.size(); ++i) {
    const unode_t *a = _roots[i].edge;
    const unode_t *b = a == lchild ? rchild : (a == rchild ? lchild : a->back);
    pos_of[a->uid] = i;
    pos_of[b->uid] = i;
  }
  auto requested = [&](const unode_t *c) {
    size_t i = pos_of[c->uid];
    return i >= begin && i < end;
  };
  // does the subtree below c, the edge above c included, hold a requested placement?
  std::vector<char> needed(n_unodes, 0);
  struct marker_t {
    const decltype(requested) &req;
    std::vector<char>         &needed;
    bool operator()(const unode_t *c) const {
      bool need = req(c);
      if (c->next) {
        bool a = (*this)(c->next->back), b = (*this)(c->next->next->back);
        need = need || a || b;
      }
      needed[c->uid] = need ? 1 : 0;
      return need;
    }
  } mark{requested, needed};
  mark(lchild);
  mark(rchild);

  struct ref_t {
    unsigned int clv;
    int          scaler;
  };
  std::vector<char> pm_seen((size_t)pm0 + 3, 0);
  auto use_pm = [&](unsigned int idx, double len) {
    if (idx < pm_seen.size() && pm_seen[idx]) return;
    if (idx < pm_seen.size()) pm_seen[idx] = 1;
    out.mi.push_back(idx);
    out.bl.push_back(len);
  };
  // close a placement: the two root half-branches and the root operation; child1 is the
  // end point root_by would make the left child (src/tree.cpp:273-320)
  auto emit_placement = [&](const unode_t *c, ref_t below, ref_t above) {
    const size_t    i = pos_of[c->uid];
    root_location_t rl = _roots[i];
    if (!ratio.empty()) rl.brlen_ratio = ratio[i];
    out.mi.push_back(ML);
    out.bl.push_back(rl.brlen());
    out.mi.push_back(MR);
    out.bl.push_back(rl.brlen_compliment());
    const bool      c_is_left = rl.edge == c;
    const ref_t     l = c_is_left ? below : above, r = c_is_left ? above : below;
    rdk_operation_t op;
    op.parent_clv_index = root_clv_index();
    op.parent_scaler_index = root_scaler_index();
    op.child1_clv_index = l.clv;
    op.child1_scaler_index = l.scaler;
    op.child1_matrix_index = ML;
    op.child2_clv_index = r.clv;
    op.child2_scaler_index = r.scaler;
    op.child2_matrix_index = MR;
    out.ops.push_back(op);
    out.pm_off.push_back((unsigned)out.mi.size());
    out.op_off.push_back((unsigned)out.ops.size());
    out.root_pos.push_back(i);
  };

  std::function<void(const unode_t *, ref_t, unsigned int, double, unsigned int)> descend;
  // c faces up; `up` is the CLV on the far side of the edge above c, directed towards c
  auto handle_edge = [&](const unode_t *c, ref_t up, unsigned int depth) {
    if (requested(c)) emit_placement(c, ref_t{c->clv_index, c->scaler_index}, up);
    descend(c, up, c->pmatrix_index, c->length, depth + 1);
  };
  descend = [&](const unode_t *c, ref_t up, unsigned int edge_pm, double edge_len, unsigned int depth) {
    if (!c->next) return;
    const unode_t *k[2] = {c->next->back, c->next->next->back};
    for (int i = 0; i < 2; ++i) {
      const unode_t *child = k[i], *sib = k[1 - i];
      if (!needed[child->uid]) continue;
      if (depth >= extra)
        throw std::runtime_error("generate_sweep_operations: the sweep needs more directed-CLV buffers "
                                 "than were set aside (sweep_depth_bound)");
      const ref_t U{clv0 + depth, scaler0 + (int)depth};
      use_pm(edge_pm, edge_len);
      use_pm(sib->pmatrix_index, sib->length);
      rdk_operation_t op;
      op.parent_clv_index = U.clv;
      op.parent_scaler_index = U.scaler;
      op.child1_clv_index = up.clv;
      op.child1_scaler_index = up.scaler;
      op.child1_matrix_index = edge_pm;
      op.child2_clv_index = sib->clv_index;
      op.child2_scaler_index = sib->scaler_index;
      op.child2_matrix_index = sib->pmatrix_index;
      out.ops.push_back(op);
      handle_edge(child, U, depth);
    }
  };

  const ref_t L{lchild->clv_index, lchild->scaler_index}, R{rchild->clv_index, rchild->scaler_index};
  if (requested(lchild)) emit_placement(lchild, L, R);
  descend(lchild, R, MC, L0, 0);
  descend(rchild, L, MC, L0, 0);
  return out;
}

void rooted_tree_t::clear_traversal_data() {
  for (auto &u : _tree->arena) u.mark = 0;
}

root_location_t rooted_tree_t::current_root() const {
  if (!rooted()) throw std::runtime_error("Failed to return root, tree is unrooted");
  return _current_rl;
}

// src/tree.cpp:443-492
std::string rooted_tree_t::newick(bool annotations) const {
  for (auto &u : _tree->arena) const_cast<unode_t &>(u).annotation.clear();
  if (annotations) {
    for (const auto &kv : _root_annotations) {
      if (kv.second.empty()) continue;
      std::string a = "[&&NHX";
      for (const auto &p : kv.second) a += ':' + p.first + '=' + p.second;
      a += ']';
      kv.first->annotation = a;
    }
  }
  auto ser = [](const unode_t *n) {
    return (n->has_label ? n->label : std::string()) + ':' + std::to_string(n->length) + n->annotation;
  };
  return rd::utree_export_newick(_tree->vroot, ser);
}

bool rooted_tree_t::branch_length_sanity_check() const {
  auto nodes = full_traverse();
  nodes.pop_back();
  std::sort(nodes.begin(), nodes.end(),
            [](unode_t *a, unode_t *b) { return a->length < b->length; });
  size_t i1 = (nodes.size() - 1) / 2, i2 = nodes.size() / 2;
  double median = (nodes[i1]->length + nodes[i2]->length) / 2.0;
  return !(median * 10.0 < nodes.back()->length || nodes.front()->length < median / 10.0);
}

void rooted_tree_t::annotate_node(size_t node_id, const std::string &k, const std::string &v) {
  annotate_node(_roots[node_id], k, v);
}
void rooted_tree_t::annotate_node(const root_location_t &rl, const std::string &k,
                                  const std::string &v) {
  annotate_node(rl.edge, k, v);
}
void rooted_tree_t::annotate_node(unode_t *n, const std::string &k, const std::string &v) {
  _root_annotations[n].emplace_back(k, v);
}
void rooted_tree_t::annotate_ratio(size_t node_id, double ratio) {
  annotate_ratio(_roots[node_id], ratio);
}
void rooted_tree_t::annotate_ratio(const root_location_t &rl, double ratio) {
  annotate_branch(rl, "alpha", std::to_string(ratio), std::to_string(1 - ratio));
}
void rooted_tree_t::annotate_lh(size_t node_index, double lh) { annotate_lh(_roots[node_index], lh); }
void rooted_tree_t::annotate_lh(const root_location_t &rl, double lh) {
  annotate_branch(rl, "LLH", std::to_string(lh));
}
void rooted_tree_t::annotate_branch(size_t node_id, const std::string &k, const std::string &v) {
  annotate_branch(_roots[node_id], k, v);
}
void rooted_tree_t::annotate_branch(const root_location_t &rl, const std::string &k,
                                    const std::string &v) {
  annotate_branch(rl, k, v, v);
}
// src/tree.cpp:739-762: the far end of the branch is the neighbour itself, or,
// when the neighbour is the two-unode virtual root, the root's other child
void rooted_tree_t::annotate_branch(const root_location_t &rl, const std::string &k,
                                    const std::string &left, const std::string &right) {
  annotate_node(rl.edge, k, left);
  size_t   ring = 0;
  unode_t *start = rl.edge->back;
  if (start->next)
    for_ring(start, [&](unode_t *) { ++ring; });
  else
    ring = 1;
  if (ring > 2)
    annotate_node(rl.edge->back, k, right);
  else
    annotate_node(rl.edge->back->next->back, k, right);
}

static void children_distance_rec(unode_t *cur, double depth, std::vector<double> &d) {
  depth += cur->length;
  if (!cur->next) {
    d.push_back(depth);
    return;
  }
  children_distance_rec(cur->next->back, depth, d);
  children_distance_rec(cur->next->next->back, depth, d);
}

std::vector<double> rooted_tree_t::get_forward_children_distance(unode_t *rl) const {
  if (!rl->next) return {0.0};
  std::vector<double> d;
  children_distance_rec(rl->next->back, 0.0, d);
  children_distance_rec(rl->next->next->back, 0.0, d);
  return d;
}

std::vector<double> rooted_tree_t::get_backward_children_distance(unode_t *rl) const {
  std::vector<double> d;
  children_distance_rec(rl->back, -rl->length, d);
  return d;
}

std::vector<std::pair<root_location_t, double>> rooted_tree_t::apply_foreach_branch_map_reduce(
    const std::function<double(double, double, double)>      &map_func,
    const std::function<double(const std::vector<double> &)> &reduce_func) const {
  // O(tips^2) pairs per branch (the reference's algorithm, src/tree.cpp:826-861): the branches are
  // independent and each keeps its own term order, so they are scored in parallel with the same
  // bits as the serial loop
  std::vector<double> score(_roots.size(), 0.0);
#pragma omp parallel for schedule(dynamic, 4)
  for (size_t r = 0; r < _roots.size(); ++r) {
    const auto         &rl = _roots[r];
    auto                fwd = get_forward_children_distance(rl.edge);
    auto                bwd = get_backward_children_distance(rl.edge);
    std::vector<double> vals;
    vals.reserve(fwd.size() * bwd.size());
    for (double f : fwd)
      for (double b : bwd) vals.push_back(map_func(f, b, rl.saved_brlen));
    score[r] = reduce_func(vals);
  }
  std::vector<std::pair<root_location_t, double>> ret;
  ret.reserve(_roots.size());
  for (size_t r = 0; r < _roots.size(); ++r) ret.emplace_back(_roots[r], score[r]);
  return ret;
}

static std::vector<root_location_t>
ranked(std::vector<std::pair<root_location_t, double>> scored) {
  std::sort(scored.begin(), scored.end(),
            [](const std::pair<root_location_t, double> &a,
               const std::pair<root_location_t, double> &b) { return a.second > b.second; });
  std::vector<root_location_t> ret;
  ret.reserve(scored.size());
  for (auto &s : scored) ret.push_back(s.first);
  return ret;
}

// src/tree.cpp:863-901
std::vector<root_location_t> rooted_tree_t::rank_midpoints() const {
  auto map = [](double l, double r, double brlen) -> double {
    if (l < r) std::swap(l, r);
    double diff = l - r;
    if (diff < brlen) {
      r += diff;
      double adj = (brlen - diff) / 2.0;
      r += adj;
      l += adj;
    } else {
      r += brlen;
    }
    double tot = r + l;
    return (1 - (diff * diff) / tot) * tot;
  };
  auto reduce = [](const std::vector<double> &v) { return *std::max_element(v.begin(), v.end()); };
  return ranked(apply_foreach_branch_map_reduce(map, reduce));
}

root_location_t rooted_tree_t::midpoint() const { return rank_midpoints().front(); }

// src/tree.cpp:907-940
std::vector<root_location_t> rooted_tree_t::rank_modified_mad() const {
  auto map = [](double l, double r, double brlen) -> double {
    double dt = l + r + brlen;
    double rho = std::min(std::max((dt - 2 * l) / (2 * brlen), 0.0), 1.0);
    l = l + rho * brlen;
    return (l / dt - 1);
  };
  auto reduce = [](const std::vector<double> &v) {
    double acc = 0.0;
    for (double x : v) acc += x * x;
    acc /= (double)v.size();
    return std::sqrt(acc);
  };
  return ranked(apply_foreach_branch_map_reduce(map, reduce));
}
