// plan_dump.cpp — the stage-8 circuit plans of csrc/host/ip_plan.h as flat int arrays, for the Python executor of
// tests/exact_stage8_ref.py.  Built by the tests with g++ into a temporary directory and loaded with ctypes; it is not part
// of the library, whose ABI does not carry the plans.
//
// Layout of plan_dump(kind, nvals): [nvals, pool_size, nin_bits, nlayers, result[16]] then per layer
//   [npre, (dst, a, b) x npre, ncbs, pool index x ncbs, nref, (pos, dst) x nref, njobs, (sel[8], lut, acc, out) x njobs,
//    npost, (dst, a, b) x npost].
#include <vector>

#include "ip_plan.h"

using namespace cbs_host;

namespace {

void put_adds(std::vector<int> &v, const std::vector<IpAdd> &adds)
{
    v.push_back((int)adds.size());
    for (const IpAdd &a : adds) v.insert(v.end(), {a.dst, a.a, a.b});
}

}  // namespace

extern "C" {

// kind 0: inner product, 1: sum, 2: maximum.  Writes min(cap, size) ints to buf and returns the size (-1: bad kind).
int plan_dump(int kind, int nvals, int *buf, int cap)
{
    if (kind < 0 || kind > 2) return -1;
    const IpPlan p = kind == 0 ? ip_make_plan(nvals) : kind == 1 ? sum_make_plan(nvals) : max_make_plan(nvals);
    std::vector<int> v = {p.nvals, p.pool_size, p.nin_bits, (int)p.layers.size()};
    v.insert(v.end(), p.result, p.result + 16);
    for (const IpLayer &L : p.layers) {
        put_adds(v, L.pre);
        v.push_back((int)L.cbs.size());
        v.insert(v.end(), L.cbs.begin(), L.cbs.end());
        v.push_back((int)L.refresh.size());
        for (const IpRefresh &r : L.refresh) v.insert(v.end(), {r.pos, r.dst});
        v.push_back((int)L.jobs.size());
        for (const IpJob &j : L.jobs) {
            v.insert(v.end(), j.sel, j.sel + 8);
            v.insert(v.end(), {j.lut, j.acc, j.out});
        }
        put_adds(v, L.post);
    }
    for (int i = 0; i < cap && i < (int)v.size(); i++) buf[i] = v[(size_t)i];
    return (int)v.size();
}

unsigned plan_lut_value(int lut, unsigned idx) { return ip_lut_value(lut, idx); }

int plan_num_luts() { return kIpNumLuts; }

}  // extern "C"
