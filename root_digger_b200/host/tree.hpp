// tree.hpp -- host-side traversal scheduler of the B200 RootDigger engine.
//
// Mirrors the interface of the reference's rooted_tree_t (src/tree.hpp:54-201)
// and of the few coraxlib utree facilities it relies on (parse, clone,
// post-order traversal, operation generation, newick export; SURVEY.md
// Appendix A-7), so that model_t can be written exactly as in the reference.
// The OUTPUT FORMAT is the contract with the device engine: an array of
// rdk_operation_t plus (pmatrix index, branch length) pairs.
//
// Pure host code, no CUDA and no likelihood arithmetic in here.
#ifndef RD_HOST_TREE_HPP_
#define RD_HOST_TREE_HPP_

#include <rdk.h>

#include <deque>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <tuple>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <vector>

namespace rd {

// One "half node" of an unrooted tree: a tip is a single unode, an inner node
// a ring of three (two for the virtual root) linked through `next`; `back`
// crosses the edge.  Field meaning follows corax_unode_t.
struct unode_t {
  unode_t     *next = nullptr;
  unode_t     *back = nullptr;
  double       length = 0.0;
  std::string  label;
  bool         has_label = false;
  unsigned int clv_index = 0;
  int          scaler_index = RDK_SCALE_BUFFER_NONE;
  unsigned int pmatrix_index = 0;
  unsigned int node_index = 0;
  int          mark = 0;          // traversal tag (the reference uses ->data)
  unsigned int uid = 0;           // position in utree_t::arena (dense key for per-unode tables)
  std::string  annotation;        // NHX text appended on export
};

struct utree_t {
  unsigned int           tip_count = 0;
  unsigned int           inner_count = 0;
  unsigned int           edge_count = 0;
  std::vector<unode_t *> nodes;  // tips first (by clv index), then one unode per inner node
  unode_t               *vroot = nullptr;
  std::deque<unode_t>    arena;  // owns every unode, addresses are stable
};

// parse a newick string; a bifurcating top level is unrooted the way
// corax_utree_parse_newick_unroot does (vroot = first top-level child with
// descendants, its `back` = the other child, the two root branches merged)
std::unique_ptr<utree_t> utree_parse_newick_string_unroot(const std::string &newick);
std::unique_ptr<utree_t> utree_parse_newick_unroot(const std::string &filename);
std::unique_ptr<utree_t> utree_clone(const utree_t &src);

// post-order traversal from vroot: subtree behind vroot->back first, then the
// other children of vroot, then vroot.  `accept` gates both emission of a node
// and descent into it.
std::vector<unode_t *> utree_traverse_postorder(unode_t *vroot,
                                                const std::function<bool(unode_t *)> &accept);

// corax_utree_create_operations on the first `count` nodes of `trav`
void utree_create_operations(const std::vector<unode_t *> &trav, size_t count,
                             std::vector<double> &branches,
                             std::vector<unsigned int> &pmatrix_indices,
                             std::vector<rdk_operation_t> &ops);

std::string utree_export_newick(const unode_t *vroot,
                                const std::function<std::string(const unode_t *)> &serialize);

}  // namespace rd

// ---------------------------------------------------------------------------
// reference-facing names (global namespace, as in src/tree.hpp)
// ---------------------------------------------------------------------------
#define GENERATE_AND_UNPACK_OPS(TREE, RL, OPS, PM, BR)                                             \
  {                                                                                                \
    auto results = TREE.generate_operations(RL);                                                   \
    OPS = std::move(std::get<0>(results));                                                         \
    PM = std::move(std::get<1>(results));                                                          \
    BR = std::move(std::get<2>(results));                                                          \
  }

// src/tree.hpp:24-50
struct root_location_t {
  rd::unode_t *edge = nullptr;
  size_t       id = 0;
  double       saved_brlen = 0.0;
  double       brlen_ratio = 0.5;

  double brlen() const { return saved_brlen * brlen_ratio; }
  double brlen_compliment() const { return saved_brlen * (1 - brlen_ratio); }
  std::string label() const { return edge->has_label ? edge->label : "(null)"; }
  bool is_internal() const { return edge->next != nullptr && edge->back->next != nullptr; }
  bool is_external() const { return !is_internal(); }
  bool operator==(const root_location_t &o) const {
    return edge == o.edge && brlen_ratio == o.brlen_ratio;
  }
  bool operator!=(const root_location_t &o) const { return !(*this == o); }
};

class rooted_tree_t {
public:
  typedef std::tuple<std::vector<rdk_operation_t>, std::vector<unsigned int>, std::vector<double>>
      op_bundle_t;

  rooted_tree_t() = default;
  explicit rooted_tree_t(const std::string &tree_filename);
  static rooted_tree_t from_newick(const std::string &newick_text);

  rooted_tree_t(rooted_tree_t &&other) noexcept;
  rooted_tree_t(const rooted_tree_t &other);
  rooted_tree_t &operator=(rooted_tree_t &&other) noexcept;
  rooted_tree_t &operator=(const rooted_tree_t &other);
  ~rooted_tree_t() = default;

  root_location_t root_location(size_t index) const;
  root_location_t root_location(const std::string &label) const;
  root_location_t root_location() const { return _current_rl; }
  // whether root_by(rl) roots the tree: on an unrooted tree whose start node is rl's edge it only
  // rewrites the lengths next to that node (update_root, src/tree.cpp:273-320)
  bool can_root_by(const root_location_t &rl) const { return rooted() || rl.edge != _tree->vroot; }

  root_location_t              midpoint() const;
  std::vector<root_location_t> rank_midpoints() const;
  std::vector<root_location_t> rank_modified_mad() const;

  size_t       root_count() const { return _roots.size(); }
  unsigned int tip_count() const { return _tree->tip_count; }
  unsigned int inner_count() const { return _tree->inner_count + 1; }
  unsigned int branch_count() const { return _tree->tip_count * 2 - 2; }
  unsigned int root_clv_index() const { return _tree->vroot->clv_index; }
  int          root_scaler_index() const { return _tree->vroot->scaler_index; }

  root_location_t                     current_root() const;
  const std::vector<root_location_t> &roots() const { return _roots; }
  std::vector<root_location_t>        internal_root_locations() const;
  std::vector<root_location_t>        external_root_locations() const;

  std::unordered_map<std::string, unsigned int> label_map() const;
  std::unordered_set<std::string>               label_set() const;

  op_bundle_t generate_operations(const root_location_t &);
  std::tuple<rdk_operation_t, std::vector<unsigned int>, std::vector<double>>
              generate_derivative_operations(const root_location_t &root);
  op_bundle_t generate_root_update_operations(const root_location_t &new_root);

  // ---- B200-first addition (no counterpart in src/tree.hpp) -------------------
  // The placement sweep of suggest_roots_lh (src/model.cpp:865-889) as ONE pre-order
  // pass over DIRECTED CLVs instead of 2n-3 move_root + compute_lh_root rounds.
  // Precondition: the tree is rooted and every inner CLV is valid for the current
  // root (compute_lh).  For the edge (v, a), a below v seen from the current root,
  //   U(a) = (P(parent edge of v) U(v)) o (P(sibling edge) D(sibling))
  // is the CLV at v directed towards a; it is exactly the CLV move_root would leave
  // in v's buffer after re-rooting on (v, a) -- same two children, same P-matrices,
  // a commutative product -- so the root log-likelihood of every placement has the
  // same bits as the reference's loop.  The U's live in `extra` spare CLV / scale
  // buffers (one per depth level: the DFS only needs the current root-to-edge
  // stack) starting at clv0 / scaler0; three spare P-matrix indices starting at
  // pm0 hold the two root half-branches and the full length of the current root
  // edge, so NOTHING the reference-shaped calls rely on is modified: the tree
  // stays rooted where it was and its CLVs, scalers and P-matrices keep their
  // values.  The output has the shape rdk_sweep_root_placements takes; the last
  // operation of each placement is the root operation.  placement q scores the
  // root at position root_pos[q] of roots(), at the ratio that root location holds
  // (0.5) or, when `ratio` is not empty, at ratio[root_pos[q]] (one entry per root
  // of roots()): the two root half-branches are then those generate_derivative_operations
  // gives for that root location at that ratio, child 1 (the location's edge) taking
  // ratio * length.
  struct sweep_schedule_t {
    std::vector<unsigned int>    pm_off{0}, op_off{0}, mi;
    std::vector<double>          bl;
    std::vector<rdk_operation_t> ops;
    std::vector<size_t>          root_pos;
  };
  // spare CLV / scale buffers generate_sweep_operations can need for ANY current root
  unsigned int     sweep_depth_bound() const;
  sweep_schedule_t generate_sweep_operations(size_t begin, size_t end, unsigned int clv0, int scaler0,
                                             unsigned int pm0, unsigned int extra,
                                             const std::vector<double> &ratio = {}) const;

  void root_by(unsigned int root_id) { root_by(_roots[root_id]); }
  void root_by(const root_location_t &);
  void update_root(root_location_t);
  void unroot();
  bool rooted() const;
  bool branch_length_sanity_check() const;
  bool sanity_check() const { return branch_length_sanity_check(); }

  std::string newick(bool annotations = true) const;
  void        clear_newick_annotations() { _root_annotations.clear(); }

  void annotate_node(const root_location_t &rl, const std::string &key, const std::string &value);
  void annotate_node(size_t node_id, const std::string &key, const std::string &value);
  void annotate_branch(size_t node_id, const std::string &key, const std::string &value);
  void annotate_branch(const root_location_t &rl, const std::string &key, const std::string &value);
  void annotate_branch(const root_location_t &rl, const std::string &key,
                       const std::string &left_value, const std::string &right_value);
  void annotate_lh(size_t node_index, double lh);
  void annotate_lh(const root_location_t &node_index, double lh);
  void annotate_ratio(size_t node_id, double ratio);
  void annotate_ratio(const root_location_t &node_index, double ratio);

  std::vector<std::pair<root_location_t, double>> apply_foreach_branch_map_reduce(
      const std::function<double(double, double, double)>      &map_func,
      const std::function<double(const std::vector<double> &)> &reduce_func) const;

  bool empty() const { return !_tree; }

private:
  void init_from_tree();
  void sort_root_locations();
  void generate_root_locations();
  void copy_from(const rooted_tree_t &other);
  void add_root_space();

  std::vector<rd::unode_t *> full_traverse() const;
  void find_path(rd::unode_t *n1, rd::unode_t *n2);
  bool find_path_recurse(rd::unode_t *n1, rd::unode_t *n2);
  void clear_traversal_data();
  void annotate_node(rd::unode_t *node, const std::string &key, const std::string &value);

  std::vector<double> get_forward_children_distance(rd::unode_t *rl) const;
  std::vector<double> get_backward_children_distance(rd::unode_t *rl) const;

  std::unique_ptr<rd::utree_t> _tree;
  rd::unode_t                 *_root_left = nullptr;   // the two spare unodes of the virtual root
  rd::unode_t                 *_root_right = nullptr;
  root_location_t              _current_rl;
  std::vector<root_location_t> _roots;
  std::unordered_map<rd::unode_t *, std::vector<std::pair<std::string, std::string>>>
       _root_annotations;
  bool _rooted = false;
};

#endif
