// gw-b200: cudaextender package header -- same names and values as the reference's
// cudaextender/include/claraparabricks/genomeworks/cudaextender/cudaextender.hpp:34-50, over the C ABI (include/gwb200.h).
#pragma once

#include "../../../gwb200.h"

#include <cstdint>

namespace claraparabricks
{
namespace genomeworks
{
namespace cudaextender
{

/// CUDA Extender status type
enum StatusType
{
    success           = 0,
    invalid_operation = 1,
    invalid_input     = 2,
    generic_error
};

/// Extension types; ungapped_xdrop performs ungapped extension with an x-drop threshold
enum ExtensionType
{
    ungapped_xdrop = 0,
};

/// Initialize CUDA Extender context (nothing to do in this engine).
inline StatusType Init() { return success; }

} // namespace cudaextender
} // namespace genomeworks
} // namespace claraparabricks
