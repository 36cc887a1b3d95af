// ahsoka_main.cpp — `Ahsoka phase` / `Ahsoka only-bubbles` with the phasing step behind the
// C ABI.  Same options, same files, same stdout banners as reference src/polyassembly.cpp:22-176.
// Built with AHSOKA_REFERENCE, the reference's own translation units (graph.cpp, alignmentreader.cpp,
// argumentparser.cpp, chainstoreadset.cpp) are linked unchanged, as BASELINE.json's north_star prescribes,
// and AHSOKA_HOST=reference runs every host stage through them; built without them, the declarations
// and the parser under standalone/ take their place and AHSOKA_HOST=reference exits with 69.  By default the stages either side of the
// phasing call that cannot ingest a BASELINE-sized input (SURVEY §8 f1, f4: GFA parsing and bubble
// detection copying node sequences at every step, the GAF reader's O(L²) strings per line, the O(B²)
// allele-path enumeration) run through this repo's result-identical replacements (graph_native.cpp,
// gaf_reader.cpp, chain_alleles.cpp), which fill the reference's own Graph object;
// tests/test_host_parity.py compares the two byte for byte.  `-t N` with N > 1 runs the
// same single batch call (the reference's two-thread experiment, polyassembly.cpp:190-222,
// only ever processed the ten largest chains and is not a parity target, SURVEY §3.3).
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <iostream>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "alignmentreader.hpp"
#include "argumentparser.hpp"
#include "graph.hpp"
#include "gaf_reader.hpp"
#include "ahsoka_b200.h"

#include <sys/stat.h>
#include <unistd.h>

using std::cerr; using std::cout; using std::endl; using std::string;
typedef std::unordered_map<int, std::unordered_map<int, std::vector<std::vector<int>>>> ChainAlleles;

ChainAlleles ChainsToReadsetDetailed(Graph graph);     // reference src/chainstoreadset.cpp:161
void alignmentsToReadset(AlignmentReader&, Graph&, ChainAlleles&, string, bool, std::vector<std::pair<int, int>>&, std::mutex&);
void alignmentsToReadset(const ahs_host::GafStore&, Graph&, ChainAlleles&, string, bool, std::vector<std::pair<int, int>>&, std::mutex&);
namespace ahs_host { int unphased_chains(); }
namespace ahs_host {
ChainAlleles chain_alleles(const Graph& graph);
int read_gfa(const std::string& filename, Graph& graph, std::string& err);
int find_bubbles(Graph& graph, std::string& err);
}

namespace {
struct StageTimer {     // AHSOKA_TIMING=1: "timing: <stage> <ms>" on stderr
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    const char* name;
    explicit StageTimer(const char* n) : name(n) {}
    ~StageTimer() {
        if (!getenv("AHSOKA_TIMING")) return;
        cerr << "timing: " << name << " " << std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() << endl;
    }
};
}

int main(int argc, char* argv[]) {
    cerr << "Ahsoka: Haplotype assembly for diploid and polyploid genomes based on HiFi and ultra-long ONT data" << endl;
    cerr << "author: Rebecca Serra Mari" << endl;
    ArgumentParser argparser;
    argparser.add_command("Ahsoka [options] -g <graph.gfa> -a <alignments.gaf>");
    argparser.add_subcommand("only-bubbles", {'g', 'o'}, {'t'});
    argparser.add_subcommand("phase", {'g', 'a', 'o'}, {'s', 't'});
    string cmd = argparser.get_subcommand(argc, argv);
    if (cmd == "phase") {
        argparser.add_mandatory_argument('g', "genome assembly graph in gfa format, e.g. by hifiasm");
        argparser.add_mandatory_argument('a', "alignments of ONT reads to the assembly graph, in gaf format");
        argparser.add_mandatory_argument('o', "output folder to store output files");
        argparser.add_optional_argument('s', "", "additional long range phasing information (StrandSeq)");
        argparser.add_optional_argument('t', "1", "number of threads to use");
    } else if (cmd == "only-bubbles") {
        argparser.add_mandatory_argument('g', "genome assembly graph in gfa format, e.g. by hifiasm");
        argparser.add_mandatory_argument('o', "output folder");
        argparser.add_optional_argument('t', "1", "number of threads to use");
    }
    argparser.add_optional_argument('k', "", "kmerfile to be written to during the kmer counting");
    argparser.add_optional_argument('c', "", "outfile for summed up unique kmer counts in short read sample");
    try { argparser.parse(argc, argv); }
    catch (const std::runtime_error& e) { argparser.print_help(); cerr << e.what() << endl; return 1; }
    catch (const std::exception& e) { return 0; }

    const string gfafile = argparser.get_arg_parameter('g');
    const string alignmentfile = argparser.get_arg_parameter('a');
    const string prefix = argparser.get_arg_parameter('o');
    const int threads = std::stoi(argparser.get_arg_parameter('t'));
    const char* host_env = getenv("AHSOKA_HOST");
    const bool ref_host = host_env && !strcmp(host_env, "reference");
    // the device context and the staging memory are set up on a second thread while the graph and the alignments are parsed
    std::thread warm;
    if (cmd == "phase") {
        struct stat sb;
        const uint64_t gaf_bytes = stat(alignmentfile.c_str(), &sb) == 0 ? (uint64_t)sb.st_size : 0;
        const char* dv = getenv("AHSOKA_DEVICE");
        const int device = dv ? atoi(dv) : 0;
        // a GAF node costs ~12 text bytes and 4 batch bytes; a pass keeps ~5.5x the node array on the device and returns ~0.6x
        warm = std::thread([=] { StageTimer t("warmup (second thread)"); ahs_warmup(device, gaf_bytes / 3 * 6, gaf_bytes / 3); });
    }
    struct Joiner { std::thread& t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{warm};
    Graph graph;
    {
        StageTimer t("read_graph");
        if (ref_host) graph = Graph::ReadGraph(gfafile);
        else {
            string err;
            if (int rc = ahs_host::read_gfa(gfafile, graph, err)) { cerr << "ahsoka_b200: " << err << endl; return rc; }   // the reference aborts on the same line
        }
    }
    cout << "number of threads used: " << threads << endl;
    cout << "threads available: " << std::thread::hardware_concurrency() << endl;
    cout << "Step 1: Graph with " << graph.nodes.size() << " nodes read" << endl;
    {
        StageTimer t("find_bubbles");
        if (ref_host) graph.findBubbles();
        else {
            string err;
            if (int rc = ahs_host::find_bubbles(graph, err)) { cerr << "ahsoka_b200: " << err << " (AHSOKA_HOST=reference runs the reference's own detection)" << endl; return rc; }
        }
    }
    cout << "Step 2: Bubbles read" << endl;
    cout << "Number of bubble chains: " << graph.chains.size() << endl;
    {
        StageTimer t("bubbleinfo");
        std::ofstream bubblefile(prefix + "-bubbleinfo.txt");
        // same bytes as polyassembly.cpp:100-110; '\n' instead of endl (one write per buffer instead of one per line)
        for (auto& chain : graph.chains) {     // graph.chains[i].id == i (graph.cpp:351-365): no getChain() scan needed
            bubblefile << "chain id: " << chain.id << "size: " << chain.bubbles.size() << '\n';
            for (auto& bubble : chain.bubbles) {
                bubblefile << "bubble id: " << bubble.id << '\n' << "node id: ";
                bubblefile << bubble.source.node_id << ",";          // Bubble::getNodes() order (graph.cpp:96-104) without copying the nodes
                for (auto& node : bubble.innerNodes) bubblefile << node.node_id << ",";
                bubblefile << bubble.sink.node_id << ",";
                bubblefile << '\n';
            }
        }
    }
    // every output file is closed by now: leave without running the destructors of the graph (tens of millions of small
    // allocations, seconds at BASELINE scale); nothing observable depends on them
    auto leave = [&]() -> int {
        if (warm.joinable()) warm.join();
        cout.flush(); cerr.flush(); fflush(nullptr);
        const int rc = ahs_host::unphased_chains() > 0 ? 3 : 0;      // a chain beyond a build limit was not phased: say so in the exit code
        _exit(rc);
        return rc;
    };
    if (cmd == "only-bubbles") return leave();

    AlignmentReader alignmentreader;
    ahs_host::GafStore store;
    int64_t n_alignment_chains;
    {
        StageTimer t("read_alignments");
        if (ref_host) {
            alignmentreader.readAlignmentfile(alignmentfile, graph);
            n_alignment_chains = (int64_t)alignmentreader.alignments.size();
        } else {
            string err;
            if (ahs_host::read_gaf(alignmentfile, graph, store, err, threads > 1 ? threads : 0)) {
                cerr << "ahsoka_b200: " << err << endl;      // the reference aborts on the same line (assert / uncaught exception)
                return 65;
            }
            n_alignment_chains = (int64_t)store.by_chain.size();
        }
    }
    cout << "Step 3: Alignments read" << endl;
    cout << "Number of alignments: " << n_alignment_chains << endl;
    ChainAlleles chainpathToAlleles;
    { StageTimer t("chain_alleles"); chainpathToAlleles = ref_host ? ChainsToReadsetDetailed(graph) : ahs_host::chain_alleles(graph); }
    cout << "Step 4: Chain paths computed " << endl;
    cout << "Number of chain paths: " << chainpathToAlleles.size() << endl;
    std::vector<std::pair<int, int>> size_sorting;
    for (auto& chainmap : chainpathToAlleles) size_sorting.emplace_back(chainmap.second.size(), chainmap.first);
    std::sort(size_sorting.begin(), size_sorting.end(), std::greater<>());
    cout << "Step 5: Phasing processed" << endl;
    cout << "single thread" << endl;
    cout << "size sorting: " << size_sorting.size() << endl;
    std::mutex g_display_mutex;
    if (ref_host) alignmentsToReadset(alignmentreader, graph, chainpathToAlleles, prefix, false, size_sorting, g_display_mutex);
    else alignmentsToReadset(store, graph, chainpathToAlleles, prefix, false, size_sorting, g_display_mutex);
    return leave();
}
