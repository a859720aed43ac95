// latok_tok5.cu -- host side of the tokenize kernel (latok_tok5.cuh): which geometry a batch runs in, its launch plan and
// the launch.  Also instantiates the kernel in the long geometry; latok_tok5_short.cu instantiates the short one.
#include "latok_tok5.cuh"
#include <stdlib.h>

namespace latok {
namespace v5 {
template int ctas_per_sm<LongGeometry>(const TableLayout &, bool, bool);
template cudaError_t launch<LongGeometry>(const Params &, int, cudaStream_t);
}  // namespace v5

template <class Geom>
static Tok5Plan plan_geometry(bool short_geometry, long long n_bytes, bool feats, const TableLayout &tl, bool is_default,
                              int n_sm)
{
    Tok5Plan t;
    t.short_geometry = short_geometry;
    t.range_bytes = Geom::RANGE;
    t.nranges = n_bytes / Geom::RANGE + 1;
    t.ntiles = (t.nranges + Geom::NW - 1) / Geom::NW;
    t.plane_words = (size_t)t.nranges * Geom::RS * NFEAT * 32;
    t.grid = n_sm * v5::ctas_per_sm<Geom>(tl, is_default, feats);
    if ((long long)t.grid > t.ntiles) t.grid = (int)t.ntiles;
    return t;
}

Tok5Plan tokenize5_plan(long long n_bytes, long long n_strings, bool feats, const TableLayout &tl, bool is_default, int n_sm)
{
    // By the average string length of the batch: short strings get the short geometry.  Token features always run in the
    // long one.  LATOK_B200_GEOMETRY=short|long overrides both (read on every call).
    bool shortg = n_bytes < 4096LL * (n_strings > 0 ? n_strings : 1);
    if (feats) shortg = false;      // the token-feature instantiation lives on registers (25 planes per lane): 96 beat 24 warps per SM
    if (const char *g = getenv("LATOK_B200_GEOMETRY")) shortg = g[0] == 's';
    return shortg ? plan_geometry<v5::ShortGeometry>(true, n_bytes, feats, tl, is_default, n_sm)
                  : plan_geometry<v5::LongGeometry>(false, n_bytes, feats, tl, is_default, n_sm);
}

cudaError_t launch_tokenize5(const Tok5Plan &plan, const Params &p, cudaStream_t s)
{
    return plan.short_geometry ? v5::launch<v5::ShortGeometry>(p, plan.grid, s) : v5::launch<v5::LongGeometry>(p, plan.grid, s);
}

}  // namespace latok
