// gaf_reader.hpp — SURVEY §8 row f1: the alignment reader of the phasing path, re-built for
// batches of millions of reads.  Result-identical replacement of
//     AlignmentReader::readAlignmentfile   (reference src/alignmentreader.cpp:69-189)
//     AlignmentPath::getRawIds             (reference src/alignmentreader.cpp:56-62)
// as far as the phasing path can observe them (the per-chain entry lists that
// alignmentsToReadset consumes, and the <gaf stem>-alignment_identities.txt side file).
//
// The reference keeps, per chain, one deep copy of the whole AlignmentPath (vector<string>) for
// EVERY node of the line that lies in the chain (alignmentreader.cpp:176-183): O(L²) strings per
// line, ~130 GB for BASELINE config 2.  Here a line is parsed once, its node ids are stored once
// as int32, and a chain lists the line once (the per-node duplicates are adjacent and change no
// result, SURVEY Appendix A#2).
#ifndef AHSOKA_B200_GAF_READER_HPP
#define AHSOKA_B200_GAF_READER_HPP
#include <cstdint>
#include <string>
#include <unordered_map>
#include <vector>

#include "graph.hpp"   // Graph::nodes → chain ids: the reference's header (-I<reference>/src) or standalone/graph.hpp

namespace ahs_host {

struct GafStore {
    // one record per GAF line the reference's reader would have accepted, in file order
    std::vector<int32_t> name_id;         // interned read name (one id per distinct name; no particular order)
    std::vector<float> identity;          // stof() of the text after the last ':' of token 16
    std::vector<int32_t> startpos, endpos;
    std::vector<int64_t> node_off{0};     // CSR into node_raw
    std::vector<int32_t> node_raw;        // raw node ids (digits of the node name), path order
    std::vector<std::string> names;       // name id → name
    // chain id → lines with ≥1 node in the chain, file order; a line equal to the previous one of
    // the chain in name, identity, start, end and node names is dropped, which is what flattening the
    // reference's container does with its per-node duplicates
    std::unordered_map<int, std::vector<int32_t>> by_chain;
    int64_t n_lines() const { return (int64_t)name_id.size(); }
};

// Parses `filename` with `threads` workers (0 = hardware concurrency) and writes the identities
// side file exactly as the reference does.  Returns 0, or a non-zero code with `err` set where the
// reference would have died on an assert / uncaught exception (malformed line).
int read_gaf(const std::string& filename, const Graph& graph, GafStore& store, std::string& err, int threads = 0);

}  // namespace ahs_host
#endif
