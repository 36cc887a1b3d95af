// standalone/argumentparser.hpp — the command-line parser interface of Ahsoka's src/argumentparser.hpp, for a build of
// the CLI without the original sources: sub-commands with mandatory and optional one-letter options, each taking a value.
#ifndef AHSOKA_B200_STANDALONE_ARGUMENTPARSER_HPP
#define AHSOKA_B200_STANDALONE_ARGUMENTPARSER_HPP
#include <map>
#include <string>
#include <vector>

class ArgumentParser {
public:
    void add_command(const std::string& usage);
    void add_subcommand(const std::string& name, std::vector<char> mandatory, std::vector<char> optional);
    std::string get_subcommand(int argc, char* argv[]);
    void add_mandatory_argument(char c, const std::string& help);
    void add_optional_argument(char c, const std::string& default_value, const std::string& help);
    // throws std::runtime_error on a wrong command line; -h prints the help and throws std::logic_error
    void parse(int argc, char* argv[]);
    void print_help() const;
    std::string get_arg_parameter(char c) const;

private:
    struct Arg { std::string help, value; bool mandatory = false; };
    struct Sub { std::vector<char> mandatory, optional; };
    std::string usage_, sub_;
    std::map<std::string, Sub> subs_;
    std::map<char, Arg> args_;
};
#endif
