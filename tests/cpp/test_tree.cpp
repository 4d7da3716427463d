// KATs of include/b200sa_tree.hpp (the C++ mirror of the reference's SuffixTree): the
// preorder of `banana` and `apple`, the reference's three properties on its own test
// strings, and from_suffix_table (runs on the GPU box; compile-checked on CPU).
#include <cstdio>
#include <string>
#include <vector>

#include "b200sa_tree.hpp"

using b200sa::Node;
using b200sa::SuffixTable;
using b200sa::SuffixTree;

#define CHECK(x) do { if (!(x)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #x); return 1; } } while (0)

struct Row {
    std::string label;
    std::vector<uint32_t> terminals;
    size_t nchildren, depth;
};

static bool same(const SuffixTree &t, const std::vector<Row> &want) {
    std::vector<Node> pre = t.root().preorder();
    if (pre.size() != want.size()) return false;
    for (size_t i = 0; i < pre.size(); i++) {
        const Node &u = pre[i];
        if (std::string(t.label(u)) != want[i].label || u.suffixes() != want[i].terminals ||
            u.children().size() != want[i].nchildren || u.depth() != want[i].depth)
            return false;
    }
    return true;
}

static bool properties(const std::string &s) {
    SuffixTable st(s);
    SuffixTree t = SuffixTree::from_suffix_table(st);
    if (t.root().leaves().size() != s.size()) return false;
    for (const Node &u : t.root().preorder())
        if (!u.has_terminals() && u.children().size() < 2) return false;
    std::vector<uint32_t> idx = t.root().suffix_indices();
    return idx == st.table();
}

int main() {
    CHECK(same(SuffixTree("banana"), {{"", {6}, 3, 0}, {"a", {5}, 1, 1}, {"na", {3}, 1, 2}, {"na", {1}, 0, 3},
                                      {"banana", {0}, 0, 1}, {"na", {4}, 1, 1}, {"na", {2}, 0, 2}}));
    CHECK(same(SuffixTree("apple"), {{"", {5}, 4, 0}, {"apple", {0}, 0, 1}, {"e", {4}, 0, 1}, {"le", {3}, 0, 1},
                                     {"p", {}, 2, 1}, {"le", {2}, 0, 2}, {"ple", {1}, 0, 2}}));
    CHECK(same(SuffixTree(""), {{"", {0}, 0, 0}}));
    CHECK(same(SuffixTree("aa"), {{"", {2}, 1, 0}, {"a", {1}, 1, 1}, {"a", {0}, 0, 2}}));
    SuffixTree b("banana");
    std::vector<Node> kids = b.root().children();
    CHECK(kids.size() == 3 && b.label(kids[2]) == "na" && kids[2].ancestors().size() == 2);
    CHECK(kids[0].suffix_indices() == (std::vector<uint32_t>{5, 3, 1}));
    for (const char *s : {"", "a", "aa", "banana", "apple", "mississippi", "\xE2\x98\x83" "abc" "\xE2\x98\x83",
                          "zzzzabczzzzzabczzzzzz"})
        CHECK(properties(s));
    bool threw = false;
    try {
        SuffixTable bad = SuffixTable::from_parts("abc", {0, 0, 1});
        SuffixTree::from_suffix_table(bad);
    } catch (const std::runtime_error &) {
        threw = true;
    }
    CHECK(threw);
    std::printf("cpp tree mirror ok\n");
    return 0;
}
