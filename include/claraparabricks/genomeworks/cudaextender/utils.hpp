// gw-b200: the cudaextender helpers of cudaextender/include/claraparabricks/genomeworks/cudaextender/utils.hpp:35-145: the
// sequence encoding, and the CSV readers of seed pairs and scored segment pairs.
#pragma once

#include "extender.hpp"
#include "../io/fasta_parser.hpp"

#include <cstdlib>
#include <fstream>
#include <stdexcept>
#include <string>
#include <vector>

namespace claraparabricks
{
namespace genomeworks
{
namespace cudaextender
{

/// Sequence encoding scheme
constexpr int8_t A_NT = 0;
constexpr int8_t C_NT = 1;
constexpr int8_t G_NT = 2;
constexpr int8_t T_NT = 3;
constexpr int8_t L_NT = 4;
constexpr int8_t N_NT = 5;
constexpr int8_t X_NT = 6;
constexpr int8_t E_NT = 7;
constexpr int8_t NUC  = 8;
constexpr int8_t NUC2 = NUC * NUC;

/// Appends the seed pairs of a CSV file with one `target_position,query_position` line per pair.
inline void parse_seed_pairs(const std::string& filepath, std::vector<SeedPair>& seed_pairs)
{
    std::ifstream in(filepath);
    if (!in.is_open())
        throw std::runtime_error("Cannot open file");
    std::string field;
    while (std::getline(in, field, ','))
    {
        SeedPair s;
        s.target_position_in_read = static_cast<position_in_read_t>(std::atoi(field.c_str()));
        std::getline(in, field);
        s.query_position_in_read = static_cast<position_in_read_t>(std::atoi(field.c_str()));
        seed_pairs.push_back(s);
    }
}

/// Appends the scored segment pairs of a CSV file with `target_position,query_position,length,score` lines.
inline void parse_scored_segment_pairs(const std::string& filepath, std::vector<ScoredSegmentPair>& scored_segment_pairs)
{
    std::ifstream in(filepath);
    if (!in.is_open())
        throw std::runtime_error("Cannot open file");
    std::string field;
    while (std::getline(in, field, ','))
    {
        ScoredSegmentPair s;
        s.start_coord.target_position_in_read = static_cast<position_in_read_t>(std::atoi(field.c_str()));
        std::getline(in, field, ',');
        s.start_coord.query_position_in_read = static_cast<position_in_read_t>(std::atoi(field.c_str()));
        std::getline(in, field, ',');
        s.length = std::atoi(field.c_str());
        std::getline(in, field);
        s.score = std::atoi(field.c_str());
        scored_segment_pairs.push_back(s);
    }
}

/// Encodes a character sequence: A C G T -> 0..3, a c g t -> L_NT, N n -> N_NT, & -> E_NT, anything else -> X_NT.
inline void encode_sequence(int8_t* dst_seq, const char* src_seq, const int32_t length)
{
    for (int32_t i = 0; i < length; i++)
    {
        switch (src_seq[i])
        {
        case 'A': dst_seq[i] = A_NT; break;
        case 'C': dst_seq[i] = C_NT; break;
        case 'G': dst_seq[i] = G_NT; break;
        case 'T': dst_seq[i] = T_NT; break;
        case '&': dst_seq[i] = E_NT; break;
        case 'n':
        case 'N': dst_seq[i] = N_NT; break;
        case 'a':
        case 'c':
        case 'g':
        case 't': dst_seq[i] = L_NT; break;
        default: dst_seq[i] = X_NT; break;
        }
    }
}

} // namespace cudaextender
} // namespace genomeworks
} // namespace claraparabricks
