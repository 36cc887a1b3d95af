// standalone/graph.hpp — the graph types of Ahsoka's src/graph.hpp as the host drop-in uses them, for a build of the
// CLI without the original sources.  Graph::nodes keeps the original's container, std::unordered_map<int, Node>: chain
// ids follow its iteration order, which depends only on the keys and the order they are inserted (graph_native.cpp).
// The original's own parsing and bubble detection (Graph::ReadGraph, findBubbles) exist only in a build against its
// sources; here they fail with a message (standalone.cpp).
#ifndef AHSOKA_B200_STANDALONE_GRAPH_HPP
#define AHSOKA_B200_STANDALONE_GRAPH_HPP
#include <cstddef>
#include <functional>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

class Node {
public:
    int node_id = -1;
    std::string sequence;
    std::vector<std::pair<int, int>> childrenleft, childrenright;      // (node id, direction: 1 = +, 0 = -)
    bool visited = false;
    int chain_id = 0, bubble_id = 0;
    Node() = default;
    Node(int id, std::string seq) : node_id(id), sequence(std::move(seq)) {}
};

struct DirectedNode {
    int id = 0;
    bool direction = false;
    DirectedNode() = default;
    DirectedNode(int i, bool d) : id(i), direction(d) {}
    bool operator==(const DirectedNode& o) const { return id == o.id && direction == o.direction; }
};

namespace std {
template <> struct hash<DirectedNode> {
    size_t operator()(const DirectedNode& d) const { return hash<long long>()(((long long)d.id << 1) | (long long)d.direction); }
};
}  // namespace std

struct DirectedEdgeHash {
    size_t operator()(const std::pair<DirectedNode, DirectedNode>& e) const {
        return std::hash<DirectedNode>()(e.first) * 1000003u ^ std::hash<DirectedNode>()(e.second);
    }
};

class Bubble {
public:
    Node source, sink;
    std::vector<Node> innerNodes;
    int id = 0;
};

class Chain {
public:
    int id = 0;
    std::vector<Bubble> bubbles;
};

class Graph {
public:
    std::unordered_map<int, Node> nodes;
    std::unordered_map<DirectedNode, std::vector<DirectedNode>> edges;
    std::unordered_map<std::pair<DirectedNode, DirectedNode>, size_t, DirectedEdgeHash> offsets;
    std::vector<Chain> chains;
    static Graph ReadGraph(const std::string& filename);
    void findBubbles();
};
#endif
