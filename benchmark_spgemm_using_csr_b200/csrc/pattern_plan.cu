// pattern_plan.cu -- host side of the diagonal-pattern mode (stage_pattern.cuh): from the offset
// sets DA, DB of the operands to the lookup tables of the kernels.
#include "pattern_plan.h"

#include <algorithm>
#include <cstring>

namespace bhb {

// Accumulator layout.  The products of one B row (A offset ja fixed, jb = 0, 1, ...) are issued by
// consecutive lanes; a shared-memory wavefront serves 32 lanes x 4 bytes, 16 x 8 or 8 x 16, so
// the outputs M[ja][jb] of each such lane group should sit in distinct banks.  Greedy colouring of
// the outputs with `nb` residues (pattern_lane_group: 32, 16 or 8) against those groups,
// then position = residue + nb * (index inside the residue class).  Conflicts that remain only
// cost replays; correctness does not depend on the layout.
static void choose_layout(int nDA, int nDB, int nD, const std::vector<unsigned char> &mlog, int nb, const long long *offs,
                          std::vector<unsigned char> &pos, int &acc_len)
{
    const int cap = 256 / nb;                       // positions stay below 256
    std::vector<std::vector<int>> sets;            // lane groups
    for (int ja = 0; ja < nDA; ++ja)
        for (int j0 = 0; j0 < nDB; j0 += nb) {
            std::vector<int> s;
            for (int jb = j0; jb < std::min(nDB, j0 + nb); ++jb) s.push_back(mlog[(size_t)ja * nDB + jb]);
            if (s.size() > 1) sets.push_back(std::move(s));
        }
    std::vector<std::vector<int>> member(nD);
    for (int si = 0; si < (int)sets.size(); ++si)
        for (int o : sets[si]) member[o].push_back(si);
    std::vector<int> res(nD, -1), cls(nb, 0), cost(nb);
    auto best_residue = [&](int o) {
        std::fill(cost.begin(), cost.end(), 0);
        for (int si : member[o])
            for (int p : sets[si])
                if (p != o && res[p] >= 0) ++cost[res[p]];
        int best = -1;
        for (int r = 0; r < nb; ++r) {
            if (cls[r] >= cap) continue;
            if (best < 0 || cost[r] < cost[best] || (cost[r] == cost[best] && cls[r] < cls[best])) best = r;
        }
        return best;
    };
    for (int o = 0; o < nD; ++o) {
        const int r = best_residue(o);
        res[o] = r;
        ++cls[r];
    }
    for (int sweep = 0; sweep < 4; ++sweep) {
        bool moved = false;
        for (int o = 0; o < nD; ++o) {
            const int cur = res[o];
            --cls[cur];
            res[o] = -1;
            const int r = best_residue(o);
            // cost[] now holds the conflicts of o with every residue
            const int take = (cost[r] < cost[cur]) ? r : cur;
            res[o] = take;
            ++cls[take];
            moved |= take != cur;
        }
        if (!moved) break;
    }
    // Second candidate family for lattice-shaped offset sets (stencils on structured grids: the offsets are
    // z*S2 + y*S1 + x).  Coordinates are recovered from the sorted offsets by peeling runs of the smallest
    // gap, level by level; then every linear colouring (x + b*y + a*z) mod nb is scored with the true
    // cost -- the sum over lane groups of the largest bank multiplicity = shared-memory wavefronts -- and
    // the best assignment (greedy included) wins.  The 27-point stencil in doubles: greedy 77, best linear
    // 54 = conflict-free (profiles/r02_notes.md).
    auto true_cost = [&](const std::vector<int> &r) {
        int total = 0;
        std::vector<int> cnt(nb);
        for (const auto &st : sets) {
            std::fill(cnt.begin(), cnt.end(), 0);
            int mx = 0;
            for (int o : st) mx = std::max(mx, ++cnt[r[o]]);
            total += mx;
        }
        return total;
    };
    if (!sets.empty() && offs && nD >= 4) {
        // coord[level][o]: position of o inside its run at that level
        std::vector<std::vector<int>> coord;
        std::vector<long long> cur(offs, offs + nD);      // sorted representatives of the current level
        std::vector<int> owner(nD);                        // element o -> index in `cur`
        for (int o = 0; o < nD; ++o) owner[o] = o;
        for (int level = 0; level < 4 && cur.size() > 1; ++level) {
            long long g = cur[1] - cur[0];
            for (size_t i = 2; i < cur.size(); ++i) g = std::min(g, cur[i] - cur[i - 1]);
            std::vector<int> run_of(cur.size()), pos_in(cur.size());
            std::vector<long long> starts;
            for (size_t i = 0; i < cur.size(); ++i) {
                if (i == 0 || cur[i] - cur[i - 1] != g) starts.push_back(cur[i]);
                run_of[i] = (int)starts.size() - 1;
                pos_in[i] = (i == 0 || cur[i] - cur[i - 1] != g) ? 0 : pos_in[i - 1] + 1;
            }
            std::vector<int> c(nD);
            for (int o = 0; o < nD; ++o) {
                c[o] = pos_in[owner[o]];
                owner[o] = run_of[owner[o]];
            }
            coord.push_back(std::move(c));
            if (starts.size() == cur.size()) break;        // no runs at this level: not a lattice
            cur.swap(starts);
        }
        if (cur.size() > 1 && coord.size() < 4) {          // whatever is left: its index is the last coordinate
            std::vector<int> c(nD);
            for (int o = 0; o < nD; ++o) c[o] = owner[o];
            coord.push_back(std::move(c));
        }
        const int nl = (int)coord.size();
        if (nl >= 2 && nl <= 4) {
            int best_cost = true_cost(res);
            std::vector<int> cand(nD), coef(nl, 0);
            long long combos = 1;
            for (int l = 1; l < nl; ++l) combos *= nb;
            if (combos <= 4096) {
                for (long long id = 0; id < combos && best_cost > (int)sets.size(); ++id) {
                    long long t = id;
                    coef[0] = 1;
                    for (int l = 1; l < nl; ++l) {
                        coef[l] = (int)(t % nb);
                        t /= nb;
                    }
                    std::vector<int> fill(nb, 0);
                    bool ok = true;
                    for (int o = 0; o < nD && ok; ++o) {
                        int v = 0;
                        for (int l = 0; l < nl; ++l) v += coef[l] * coord[l][o];
                        cand[o] = v % nb;
                        ok = ++fill[cand[o]] <= cap;
                    }
                    if (!ok) continue;
                    const int c = true_cost(cand);
                    if (c < best_cost) {
                        best_cost = c;
                        res = cand;
                    }
                }
            }
        }
    }
    std::vector<int> next(nb, 0);
    pos.assign(nD, 0);
    int maxcls = 1;
    for (int o = 0; o < nD; ++o) {
        pos[o] = (unsigned char)(res[o] + nb * next[res[o]]);
        maxcls = std::max(maxcls, ++next[res[o]]);
    }
    acc_len = nb * maxcls;
    if (acc_len < 32) acc_len = 32;
}

bool build_pattern_plan(const int *offsA, int nA, const int *offsB, int nB, int value_size, PatternPlan &plan)
{
    plan.valid = false;
    if (nA <= 0 || nB <= 0 || nA > PAT_MAX_OFFS || nB > PAT_MAX_OFFS) return false;
    std::vector<int> DA(offsA, offsA + nA), DB(offsB, offsB + nB);
    std::sort(DA.begin(), DA.end());
    std::sort(DB.begin(), DB.end());
    if (plan.DA == DA && plan.DB == DB && plan.value_size == value_size && !plan.blob.empty()) {
        plan.valid = true;   // same patterns as the previous call: tables are already on the device
        plan.reused = true;
        return true;
    }
    std::vector<long long> sums;
    sums.reserve((size_t)nA * nB);
    for (int a : DA)
        for (int b : DB) sums.push_back((long long)a + b);
    std::sort(sums.begin(), sums.end());
    sums.erase(std::unique(sums.begin(), sums.end()), sums.end());
    const int nD = (int)sums.size();
    if (nD > PAT_MAX_OUT) return false;
    int nw = (nD + 31) / 32;
    nw = nw <= 1 ? 1 : nw <= 2 ? 2 : nw <= 4 ? 4 : 8;
    plan.DA = DA;
    plan.DB = DB;
    plan.value_size = value_size;
    plan.nD = nD;
    plan.nw = nw;
    plan.reused = false;
    std::vector<unsigned char> mlog((size_t)nA * nB), mphys((size_t)nA * nB), pos;
    std::vector<unsigned> pfull((size_t)nA * nw, 0u);
    for (int ja = 0; ja < nA; ++ja)
        for (int jb = 0; jb < nB; ++jb) {
            const long long s = (long long)DA[ja] + DB[jb];
            const int o = (int)(std::lower_bound(sums.begin(), sums.end(), s) - sums.begin());
            mlog[(size_t)ja * nB + jb] = (unsigned char)o;
            pfull[(size_t)ja * nw + (o >> 5)] |= 1u << (o & 31);
        }
    if (value_size > 0) {
        choose_layout(nA, nB, nD, mlog, pattern_lane_group(value_size), sums.data(), pos, plan.acc_len);
    } else {   // structure only: k_pat_emit writes the columns from the output masks, there is no accumulator
        pos.assign(nD, 0);
        plan.acc_len = 0;
    }
    for (size_t i = 0; i < mlog.size(); ++i) mphys[i] = pos[mlog[i]];
    // blob: byte tables first, then the 4-byte tables (aligned)
    const size_t nM = (size_t)nA * nB;
    plan.off_mphys = 0;
    plan.off_mlog = nM;
    plan.off_pos = 2 * nM;
    size_t o4 = (2 * nM + nD + 15) & ~(size_t)15;
    plan.off_pfull = o4;
    o4 += (size_t)nA * nw * 4;
    plan.off_dcol = o4;
    o4 += (size_t)nD * 4;
    plan.off_offsA = o4;
    o4 += (size_t)nA * 4;
    plan.off_offsB = o4;
    o4 += (size_t)nB * 4;
    plan.blob.assign(o4, 0);
    memcpy(plan.blob.data() + plan.off_mphys, mphys.data(), nM);
    memcpy(plan.blob.data() + plan.off_mlog, mlog.data(), nM);
    memcpy(plan.blob.data() + plan.off_pos, pos.data(), nD);
    memcpy(plan.blob.data() + plan.off_pfull, pfull.data(), pfull.size() * 4);
    std::vector<int> dcol(nD);
    for (int i = 0; i < nD; ++i) dcol[i] = (int)sums[i];   // (wraps only for sums no row can produce)
    memcpy(plan.blob.data() + plan.off_dcol, dcol.data(), (size_t)nD * 4);
    memcpy(plan.blob.data() + plan.off_offsA, DA.data(), (size_t)nA * 4);
    memcpy(plan.blob.data() + plan.off_offsB, DB.data(), (size_t)nB * 4);
    plan.valid = true;
    return true;
}

PatTables pattern_tables(const PatternPlan &plan, const unsigned char *dev_blob)
{
    PatTables t;
    t.mphys = dev_blob + plan.off_mphys;
    t.mlog = dev_blob + plan.off_mlog;
    t.pos = dev_blob + plan.off_pos;
    t.pfull = reinterpret_cast<const unsigned *>(dev_blob + plan.off_pfull);
    t.dcol = reinterpret_cast<const int *>(dev_blob + plan.off_dcol);
    t.offsA = reinterpret_cast<const int *>(dev_blob + plan.off_offsA);
    t.offsB = reinterpret_cast<const int *>(dev_blob + plan.off_offsB);
    t.nDA = (int)plan.DA.size();
    t.nDB = (int)plan.DB.size();
    t.nD = plan.nD;
    t.nw = plan.nw;
    t.acc_len = plan.acc_len;
    t.fullB = t.nDB >= 64 ? ~0ull : ((1ull << t.nDB) - 1ull);
    t.fullbits = nullptr;
    return t;
}

}  // namespace bhb
