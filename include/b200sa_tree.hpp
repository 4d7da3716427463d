// b200sa_tree.hpp -- C++ host-side mirror of the reference's `SuffixTree` / `Node`
// (suffix_tree/src/lib.rs) above b200sa_suffix_tree of b200sa.h.
//
// The tree is built on the GPU and held as six u32 arrays indexed by preorder id
// (children in first-byte order); a Node is a (tree, id) handle with the reference's
// methods.  Labels and terminals follow from the table: label(u) = text[sa[lo] +
// depth(parent), sa[lo] + depth(u)); u has a terminal iff depth(u) == n - sa[lo]
// (the root: suffix n, empty label).  A failing call throws std::runtime_error; a
// text above B200SA_TREE_MAX_N bytes throws std::length_error.
#pragma once
#include <cstdint>
#include <mutex>
#include <stdexcept>
#include <string>
#include <string_view>
#include <vector>

#include "b200sa.h"
#include "b200sa_table.hpp"

namespace b200sa {

class SuffixTree;

class Node {
  public:
    Node(const SuffixTree *t, uint32_t id) : t_(t), id_(id) {}
    uint32_t id() const { return id_; }
    bool operator==(const Node &o) const { return t_ == o.t_ && id_ == o.id_; }
    bool operator!=(const Node &o) const { return !(*this == o); }

    std::vector<Node> children() const;      // first-byte order
    std::vector<Node> ancestors() const;     // self ... root
    std::vector<Node> preorder() const;      // self and its subtree, lexicographic
    std::vector<Node> leaves() const;        // preorder nodes with terminals and a non-empty label
    std::vector<uint32_t> suffix_indices() const;   // table[lo, hi), suffix order
    uint32_t len() const;                    // size of the path label into this node
    size_t depth() const;                    // number of ancestors, not including self
    bool has_terminals() const { return !suffixes().empty(); }
    std::vector<uint32_t> suffixes() const;

  private:
    const SuffixTree *t_;
    uint32_t id_;
};

class SuffixTree {
  public:
    // SuffixTree::new: SA, LCP and the tree on the device
    explicit SuffixTree(std::string text) : text_(std::move(text)) { build(false); }
    // SuffixTree::from_suffix_table: the table is checked to be a permutation
    static SuffixTree from_suffix_table(const SuffixTable &st) { return SuffixTree(st.text(), st.table()); }

    const std::string &text() const { return text_; }
    Node root() const { return Node(this, 0); }
    std::string_view label(const Node &node) const {
        uint32_t u = node.id();
        if (u == 0) return {};
        uint32_t s = sa_[lo_[u]];
        return std::string_view(text_).substr(s + depth_[parent_[u]], depth_[u] - depth_[parent_[u]]);
    }
    size_t num_nodes() const { return parent_.size(); }
    const std::vector<uint32_t> &table() const { return sa_; }

  private:
    friend class Node;
    SuffixTree(std::string text, std::vector<uint32_t> table) : text_(std::move(text)), sa_(std::move(table)) {
        build(true);
    }
    void build(bool sa_given) {
        uint64_t n = text_.size();
        if (n > B200SA_TREE_MAX_N) throw std::length_error("SuffixTree: text longer than 2^31-1 bytes");
        size_t cap = n ? 2 * n : 1;
        sa_.resize(n);
        for (auto *v : {&parent_, &depth_, &lo_, &hi_, &end_, &nch_}) v->resize(cap);
        b200sa_tree h{parent_.data(), depth_.data(), lo_.data(), hi_.data(), end_.data(), nch_.data()};
        uint64_t k = 0;
        Context &c = Context::default_context();
        std::lock_guard<std::mutex> lk(c.mutex());
        int rc = b200sa_suffix_tree(c.get(), reinterpret_cast<const uint8_t *>(text_.data()), n, sa_.data(),
                                    sa_given ? 1 : 0, &h, &k);
        if (rc != B200SA_OK)
            throw std::runtime_error(std::string("b200sa: ") + b200sa_strerror(rc) + ": " + b200sa_last_error(c.get()));
        for (auto *v : {&parent_, &depth_, &lo_, &hi_, &end_, &nch_}) v->resize(k);
    }
    std::string text_;
    std::vector<uint32_t> sa_, parent_, depth_, lo_, hi_, end_, nch_;
};

inline std::vector<Node> Node::children() const {
    std::vector<Node> out;
    out.reserve(t_->nch_[id_]);
    for (uint32_t c = id_ + 1; c < t_->end_[id_]; c = t_->end_[c]) out.emplace_back(t_, c);
    return out;
}
inline std::vector<Node> Node::ancestors() const {
    std::vector<Node> out;
    for (uint32_t u = id_; u != 0xFFFFFFFFu; u = t_->parent_[u]) out.emplace_back(t_, u);
    return out;
}
inline std::vector<Node> Node::preorder() const {
    std::vector<Node> out;
    for (uint32_t u = id_; u < t_->end_[id_]; u++) out.emplace_back(t_, u);
    return out;
}
inline std::vector<Node> Node::leaves() const {
    std::vector<Node> out;
    for (const Node &u : preorder())
        if (u.len() > 0 && u.has_terminals()) out.push_back(u);
    return out;
}
inline std::vector<uint32_t> Node::suffix_indices() const {
    return std::vector<uint32_t>(t_->sa_.begin() + t_->lo_[id_], t_->sa_.begin() + t_->hi_[id_]);
}
inline uint32_t Node::len() const { return id_ == 0 ? 0 : t_->depth_[id_] - t_->depth_[t_->parent_[id_]]; }
inline size_t Node::depth() const { return ancestors().size() - 1; }
inline std::vector<uint32_t> Node::suffixes() const {
    uint32_t n = (uint32_t)t_->text_.size();
    if (id_ == 0) return {n};
    uint32_t s = t_->sa_[t_->lo_[id_]];
    if (t_->depth_[id_] == n - s) return {s};
    return {};
}

}  // namespace b200sa
