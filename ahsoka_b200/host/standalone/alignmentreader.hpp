// standalone/alignmentreader.hpp — the alignment types of Ahsoka's src/alignmentreader.hpp as the host drop-in uses
// them, for a build of the CLI without the original sources.  The CLI reads GAF files with ahs_host::read_gaf; the
// original's reader (AlignmentReader::readAlignmentfile) exists only in a build against its sources.
#ifndef AHSOKA_B200_STANDALONE_ALIGNMENTREADER_HPP
#define AHSOKA_B200_STANDALONE_ALIGNMENTREADER_HPP
#include <string>
#include <unordered_map>
#include <vector>

#include "graph.hpp"

class AlignmentPath {
public:
    std::string name;
    float id = 0.0f;
    int startpos = 0, endpos = 0;
    std::vector<std::string> nodes;
    std::vector<int> getRawIds();
};

class AlignmentReader {
public:
    std::unordered_map<int, std::vector<AlignmentPath>> alignments;
    void readAlignmentfile(const std::string& filename, Graph& graph);
};
#endif
