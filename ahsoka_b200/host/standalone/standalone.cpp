// standalone.cpp — what a build of the CLI without the original Ahsoka sources links instead of them: the command-line
// parser, and the original's host stages (selected with AHSOKA_HOST=reference), which fail with a message here.
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <unordered_map>

#include "alignmentreader.hpp"
#include "argumentparser.hpp"
#include "graph.hpp"

namespace {
[[noreturn]] void no_reference_host(const char* what) {
    std::cerr << "ahsoka_b200: " << what << " is the original Ahsoka's and this binary was built without its sources "
              << "(AHSOKA_HOST=reference needs a build with AHSOKA_REFERENCE set)" << std::endl;
    std::exit(69);
}
}  // namespace

Graph Graph::ReadGraph(const std::string&) { no_reference_host("Graph::ReadGraph"); }
void Graph::findBubbles() { no_reference_host("Graph::findBubbles"); }
std::vector<int> AlignmentPath::getRawIds() { no_reference_host("AlignmentPath::getRawIds"); }
void AlignmentReader::readAlignmentfile(const std::string&, Graph&) { no_reference_host("AlignmentReader::readAlignmentfile"); }
std::unordered_map<int, std::unordered_map<int, std::vector<std::vector<int>>>> ChainsToReadsetDetailed(Graph) {
    no_reference_host("ChainsToReadsetDetailed");
}

void ArgumentParser::add_command(const std::string& usage) { usage_ = usage; }

void ArgumentParser::add_subcommand(const std::string& name, std::vector<char> mandatory, std::vector<char> optional) {
    subs_[name] = Sub{std::move(mandatory), std::move(optional)};
}

std::string ArgumentParser::get_subcommand(int argc, char* argv[]) {
    sub_ = argc > 1 ? argv[1] : "";
    return sub_;
}

void ArgumentParser::add_mandatory_argument(char c, const std::string& help) {
    Arg& a = args_[c];
    a.help = help; a.mandatory = true;
}

void ArgumentParser::add_optional_argument(char c, const std::string& default_value, const std::string& help) {
    Arg& a = args_[c];
    a.help = help; a.value = default_value; a.mandatory = false;
}

void ArgumentParser::parse(int argc, char* argv[]) {
    auto sub = subs_.find(sub_);
    if (sub == subs_.end()) throw std::runtime_error("unknown sub-command '" + sub_ + "' (phase, only-bubbles)");
    auto allowed = [&](char c) {
        for (char m : sub->second.mandatory) if (m == c) return true;
        for (char o : sub->second.optional) if (o == c) return true;
        return false;
    };
    std::unordered_map<char, bool> seen;
    for (int i = 2; i < argc; i++) {
        const std::string s = argv[i];
        if (s == "-h") { print_help(); throw std::logic_error("help"); }
        if (s.size() < 2 || s[0] != '-') throw std::runtime_error("unexpected argument '" + s + "'");
        const char c = s[1];
        auto a = args_.find(c);
        if (a == args_.end()) throw std::runtime_error(std::string("unknown option -") + c);
        std::string value;
        if (s.size() > 2) value = s.substr(2);
        else if (i + 1 < argc) value = argv[++i];
        else throw std::runtime_error(std::string("option -") + c + " needs a value");
        if (!allowed(c)) continue;                      // registered, but not an option of this sub-command: ignored
        a->second.value = value;
        seen[c] = true;
    }
    for (char m : sub->second.mandatory)
        if (!seen.count(m)) throw std::runtime_error(std::string("missing mandatory option -") + m);
}

void ArgumentParser::print_help() const {
    std::cerr << "usage: " << usage_ << std::endl;
    for (auto& s : subs_) {
        std::cerr << "  " << s.first << ":";
        for (char m : s.second.mandatory) std::cerr << " -" << m;
        for (char o : s.second.optional) std::cerr << " [-" << o << "]";
        std::cerr << std::endl;
    }
    for (auto& a : args_) std::cerr << "  -" << a.first << "  " << a.second.help << std::endl;
}

std::string ArgumentParser::get_arg_parameter(char c) const {
    auto a = args_.find(c);
    return a == args_.end() ? "" : a->second.value;
}
