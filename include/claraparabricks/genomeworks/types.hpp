// gw-b200: the index types of the reference's common/base/include/claraparabricks/genomeworks/types.hpp:37-46 that callers of
// the kept API use (cudaextender's SeedPair positions, FastaParser ids).
#pragma once

#include <cstdint>

namespace claraparabricks
{
namespace genomeworks
{

/// unique ID of a read
using read_id_t = std::uint32_t;
/// number of reads
using number_of_reads_t = read_id_t;
/// position of a basepair in a read
using position_in_read_t = std::uint32_t;
/// number of basepairs
using number_of_basepairs_t = position_in_read_t;

} // namespace genomeworks
} // namespace claraparabricks
