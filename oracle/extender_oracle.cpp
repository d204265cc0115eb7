// TEST INFRASTRUCTURE ONLY: sequential restatement of the ungapped X-drop extender (cudaextender, SegAlign's ungapped
// extender; reference kernel cudaextender/src/ungapped_xdrop_kernels.cu:37-505, host pipeline ungapped_xdrop.cu:96-179).
// One seed at a time, one position at a time, exactly the rules DESIGN.md section 4 lists:
//   right extension over p = 0, 1, ... of (T[t+p], Q[q+p]), best (0, -1); left over p = 1, 2, ... of (T[t-p], Q[q-p]), best
//   (0, 0); the best moves on a strictly larger running sum; stop at the first p with max(best, max S) - S(p) > xdrop
//   (excluded) or at the first position outside a sequence;
//   entropy correction for thr <= total <= 3 thr, from the matching A/C/G/T counts over [-lp, rp] when they sum to >= 20;
//   stable sort by ((uint32)(t - q), t, length desc, score desc), then drop every element that lies on its sorted
//   predecessor's diagonal and contains or is contained in it (thrust::unique_copy compares with the predecessor).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

namespace
{

struct Ssp
{
    uint32_t query;
    uint32_t target;
    int32_t length;
    int32_t score;
};

struct Side
{
    int32_t score;
    int64_t pos;
};

// Positions p = first, first + 1, ... while p - first < n_valid; offsets t + dir * p, q + dir * p.
Side extend(const int8_t* T, const int8_t* Q, const int32_t* M, int64_t t, int64_t q, int dir, int64_t first, int64_t n_valid, int32_t xdrop)
{
    Side best{0, first - 1};
    int32_t S     = 0;
    int32_t max_s = 0; // max(best, max of S so far) == best.score: best only grows
    for (int64_t p = first; p - first < n_valid; p++)
    {
        const int tc = T[t + dir * p] & 7;
        const int qc = Q[q + dir * p] & 7;
        S            = static_cast<int32_t>(static_cast<uint32_t>(S) + static_cast<uint32_t>(M[tc * 8 + qc]));
        if (static_cast<int32_t>(static_cast<uint32_t>(std::max(max_s, S)) - static_cast<uint32_t>(S)) > xdrop)
            break;
        if (S > best.score)
        {
            best.score = S;
            best.pos   = p;
        }
        max_s = std::max(max_s, S);
    }
    return best;
}

// ln(4) in f32 as the reference computes it under -use_fast_math: lg2.approx(4) * 0.693147182f
double ln4_f32()
{
    const uint32_t bits = 0x3FB17218u;
    float f;
    std::memcpy(&f, &bits, 4);
    return static_cast<double>(f);
}

bool less_ssp(const Ssp& x, const Ssp& y)
{
    const uint32_t dx = x.target - x.query, dy = y.target - y.query;
    if (dx != dy)
        return dx < dy;
    if (x.target != y.target)
        return x.target < y.target;
    if (x.length != y.length)
        return x.length > y.length;
    return x.score > y.score;
}

bool diagonal_overlap(const Ssp& x, const Ssp& y)
{
    if (x.target - x.query != y.target - y.query)
        return false;
    const uint32_t xe = x.target + static_cast<uint32_t>(x.length);
    const uint32_t ye = y.target + static_cast<uint32_t>(y.length);
    return (x.target >= y.target && xe <= ye) || (y.target >= x.target && ye <= xe);
}

} // namespace

extern "C" {

// seeds: n pairs {query, target}; out: up to n records {query, target, length, score}; returns the number written.
// stats (may be NULL): [0] segments that passed the threshold before deduplication, [1] positions scored.
int64_t oracle_extender_run(const int8_t* query, int32_t query_length, const int8_t* target, int32_t target_length, const int32_t* score_mat,
                            int32_t xdrop, int32_t no_entropy, int32_t score_threshold, const uint32_t* seeds, int32_t n, int32_t* out,
                            int64_t* stats)
{
    std::vector<Ssp> kept;
    int64_t positions = 0;
    const int64_t tlen = target_length, qlen = query_length;
    for (int32_t s = 0; s < n; s++)
    {
        const int64_t q = seeds[2 * s], t = seeds[2 * s + 1];
        const int64_t n_right = std::max<int64_t>(0, std::min(tlen - t, qlen - q));
        const int64_t n_left  = (t > tlen || q > qlen) ? 0 : std::min(t, q);
        const Side r          = extend(target, query, score_mat, t, q, 1, 0, n_right, xdrop);
        const Side l          = extend(target, query, score_mat, t, q, -1, 1, n_left, xdrop);
        positions += n_right + n_left; // upper bound; the kernel's count is reported by the engine
        const int64_t rp    = r.pos, lp = l.pos;
        const int32_t total = static_cast<int32_t>(static_cast<uint32_t>(r.score) + static_cast<uint32_t>(l.score));
        double entropy      = 1.0;
        const int32_t thr3  = static_cast<int32_t>(3u * static_cast<uint32_t>(score_threshold));
        if (!no_entropy && total >= score_threshold && total <= thr3)
        {
            int64_t c[4] = {0, 0, 0, 0};
            for (int64_t k = -lp; k <= rp; k++)
            {
                const int8_t a = target[t + k], b = query[q + k];
                if (a == b && a >= 0 && a < 4)
                    c[a]++;
            }
            if (c[0] + c[1] + c[2] + c[3] >= 20)
            {
                const double denom = static_cast<double>(static_cast<int32_t>(rp + lp + 1));
                double acc         = 0.0;
                for (int i = 0; i < 4; i++)
                {
                    if (c[i] != 0)
                    {
                        const double p = static_cast<double>(c[i]) / denom;
                        acc            = std::fma(p, std::log(p), acc);
                    }
                }
                entropy = -acc / ln4_f32();
            }
        }
        const int32_t score = static_cast<int32_t>(static_cast<double>(total) * entropy);
        if (score >= score_threshold)
            kept.push_back(Ssp{static_cast<uint32_t>(q - lp), static_cast<uint32_t>(t - lp), static_cast<int32_t>(rp + lp), score});
    }
    std::stable_sort(kept.begin(), kept.end(), less_ssp);
    int64_t m = 0;
    for (size_t i = 0; i < kept.size(); i++)
    {
        if (i > 0 && diagonal_overlap(kept[i - 1], kept[i]))
            continue;
        out[4 * m + 0] = static_cast<int32_t>(kept[i].query);
        out[4 * m + 1] = static_cast<int32_t>(kept[i].target);
        out[4 * m + 2] = kept[i].length;
        out[4 * m + 3] = kept[i].score;
        m++;
    }
    if (stats)
    {
        stats[0] = static_cast<int64_t>(kept.size());
        stats[1] = positions;
    }
    return m;
}

} // extern "C"
