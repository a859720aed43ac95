// latok_tok5_short.cu -- the tokenize kernel (latok_tok5.cuh) in the short-string geometry, compiled in parallel with
// latok_tok5.cu.
#include "latok_tok5.cuh"

namespace latok {
namespace v5 {
template int ctas_per_sm<ShortGeometry>(const TableLayout &, bool, bool);
template cudaError_t launch<ShortGeometry>(const Params &, int, cudaStream_t);
}  // namespace v5
}  // namespace latok
