// gw-b200: io::FastaParser / create_kseq_fasta_parser (common/io/include/claraparabricks/genomeworks/io/fasta_parser.hpp:34-72)
// over a small plain-text FASTA reader (multi-line records; no compressed input, no kseq).
#pragma once

#include "../types.hpp"

#include <algorithm>
#include <fstream>
#include <memory>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

namespace claraparabricks
{
namespace genomeworks
{
namespace io
{

/// One record: the name (header line without '>', up to the first blank) and the sequence.
typedef struct
{
    std::string name;
    std::string seq;
} FastaSequence;

class FastaParser
{
public:
    virtual ~FastaParser() = default;
    /// Number of sequences kept.
    virtual number_of_reads_t get_num_seqences() const = 0;
    /// Sequence by index; std::out_of_range past the end.
    virtual const FastaSequence& get_sequence_by_id(read_id_t sequence_id) const = 0;
};

namespace details
{
class FastaParserPlain : public FastaParser
{
public:
    FastaParserPlain(const std::string& path, number_of_basepairs_t min_sequence_length, bool shuffle)
    {
        std::ifstream in(path);
        if (!in.good())
            throw std::invalid_argument("Cannot open file " + path);
        std::string line;
        bool have = false;
        FastaSequence cur;
        auto flush = [&]() {
            if (have && cur.seq.size() >= min_sequence_length)
                seqs_.push_back(cur);
            cur  = FastaSequence();
            have = false;
        };
        while (std::getline(in, line))
        {
            if (!line.empty() && line.back() == '\r')
                line.pop_back();
            if (!line.empty() && line[0] == '>')
            {
                flush();
                have     = true;
                cur.name = line.substr(1, line.find_first_of(" \t") == std::string::npos ? std::string::npos : line.find_first_of(" \t") - 1);
            }
            else if (have)
            {
                cur.seq += line;
            }
        }
        flush();
        if (shuffle)
        {
            std::mt19937 rng(0);
            std::shuffle(seqs_.begin(), seqs_.end(), rng);
        }
    }
    number_of_reads_t get_num_seqences() const override { return static_cast<number_of_reads_t>(seqs_.size()); }
    const FastaSequence& get_sequence_by_id(read_id_t sequence_id) const override { return seqs_.at(sequence_id); }

private:
    std::vector<FastaSequence> seqs_;
};
} // namespace details

/// Reads every record of `fasta_file` that is at least min_sequence_length long; shuffle = true reorders them (fixed seed).
inline std::unique_ptr<FastaParser> create_kseq_fasta_parser(const std::string& fasta_file, number_of_basepairs_t min_sequence_length = 0,
                                                             bool shuffle = true)
{
    return std::unique_ptr<FastaParser>(new details::FastaParserPlain(fasta_file, min_sequence_length, shuffle));
}

} // namespace io
} // namespace genomeworks
} // namespace claraparabricks
