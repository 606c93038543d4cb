// Work partition of the fused residual-stack kernel (fused.cu): equal-cost contiguous pieces of the (utterance, chunk)
// line, one per team of G CTAs.  Host-only plain C++ (no CUDA types), so it also builds into a CPU test driver.
#pragma once
#include <algorithm>
#include <vector>

namespace fused {

constexpr int kMaxSeg = 8;                      // segments (utterance pieces) per team

// One piece of one utterance: rows [t_start, t_out) are warm-up (they rebuild the history rings, outputs discarded),
// rows [t_out, t_end) are outputs.
struct Seg { int b, t_start, t_out, t_end; };

// segs [teams][kMaxSeg], nseg [teams]; teams == 0: no team size fits the batch (fused_max_batch)
struct Partition { std::vector<Seg> segs; std::vector<int> nseg; int teams = 0, G = 0; double cost = 0; };

// warm_cost[k] = cost (in full chunks) of the k warm-up chunks nearest the first output row: a warm-up chunk skips the skip
// GEMM and the head and runs only the layers inside the dependency cone (k_fused: rsuf[l+1] > dist); a fixed part per chunk
// (front conv, conditioning loads, chunk barrier) plus a part proportional to the layers it runs.
// Outputs start at row out0 of each utterance (0 for a one-call launch; the history length of a student stream call, whose
// rows before out0 are carried inputs): the output rows are cut into chunks counted from out0, an utterance's first piece
// starts at row 0 and warms up over rows [0, out0), later pieces warm up as usual, clamped at row 0.
inline bool try_partition(int B, int T, int out0, int kChunk, const std::vector<double>& warm_cost, int teams, double budget,
                          Partition* out) {
  const int warm_chunks = (int)warm_cost.size() - 1;
  const int NC = (T - out0 + kChunk - 1) / kChunk;
  const int lead = std::min(warm_chunks, (out0 + kChunk - 1) / kChunk);   // warm-up of the first piece (cost model only)
  std::vector<Seg> segs((size_t)teams * kMaxSeg);
  std::vector<int> nseg(teams, 0);
  int tm = 0;
  double used = 0;
  for (int b = 0; b < B; b++) {
    int c0 = 0;
    while (c0 < NC) {
      if (tm >= teams) return false;
      const int t_out = out0 + c0 * kChunk;
      const int warm = c0 == 0 ? lead : std::min(warm_chunks, (t_out + kChunk - 1) / kChunk);
      const double room = budget - used - warm_cost[warm];
      int take = room >= NC - c0 ? NC - c0 : (int)std::max(room, 0.0);   // the rest of the utterance fits, or part of it
      if (take < 1 || nseg[tm] >= kMaxSeg) {
        if (used == 0 && nseg[tm] < kMaxSeg) take = 1; else { tm++; used = 0; continue; }
      }
      Seg s;
      s.b = b; s.t_start = c0 == 0 ? 0 : std::max(0, t_out - warm * kChunk); s.t_out = t_out;
      s.t_end = std::min(T, out0 + (c0 + take) * kChunk);
      segs[(size_t)tm * kMaxSeg + nseg[tm]++] = s;
      used += take + warm_cost[warm];
      c0 += take;
    }
  }
  if (out) { out->segs.swap(segs); out->nseg.swap(nseg); out->teams = teams; }
  return true;
}

// Smallest budget (per team) that try_partition meets, to 24 bisection steps.  Needs teams * kMaxSeg >= B: a budget of
// k whole utterances with their largest warm-up, k = ceil(B / teams) <= kMaxSeg, always succeeds (a team then takes k
// whole utterances, or the rest of a split one plus k - 1 whole ones and at most one more piece), so the search for a
// first feasible budget stops there.
inline Partition partition_for(int B, int T, int out0, int kChunk, const std::vector<double>& warm_cost, int teams) {
  const int warm_chunks = (int)warm_cost.size() - 1;
  const int NC = (T - out0 + kChunk - 1) / kChunk;
  const long long total = (long long)B * NC;
  const int k = (B + teams - 1) / teams;
  const double cap = k * (NC + warm_cost[warm_chunks]) + 1;
  double lo = (double)total / teams, hi = lo + warm_chunks + 2;
  Partition best;
  while (!try_partition(B, T, out0, kChunk, warm_cost, teams, hi, &best)) {
    if (hi >= cap) return Partition();           // not reached when teams * kMaxSeg >= B
    hi *= 1.5;
  }
  for (int it = 0; it < 24; it++) {
    const double mid = 0.5 * (lo + hi);
    Partition cand;
    if (try_partition(B, T, out0, kChunk, warm_cost, teams, mid, &cand)) { hi = mid; best = cand; } else lo = mid;
  }
  best.cost = hi;
  return best;
}

// Utterances one fused launch takes on `grid` SMs: every utterance needs a segment of its own, a team holds kMaxSeg, and
// there are at most `grid` teams (G = 1).
inline long long fused_max_batch(int grid) { return (long long)grid * kMaxSeg; }

// Team size: a team of G CTAs walks its piece as a wavefront, member j+1 about `kLagLayers` layers behind member j, so
// (a) a piece costs (chunks + warm-up) / G per member, (b) the wavefront fills and drains over (G-1) lags, (c) member 0
// can only start its next chunk when member G-1 is through the same layer of the previous one: a chunk period is at
// least G lags.  Larger G shares the mid-utterance warm-up between more CTAs.  A team size leaves grid / G teams, which
// hold at most kMaxSeg utterances each: sizes with too few teams for B are not candidates.  `force_G` > 0 overrides the
// choice; a forced size with too few teams gives way to the largest one that has enough.  Returns teams == 0 when even
// G = 1 has too few (B > fused_max_batch(grid)).
constexpr double kLagLayers = 1.5;
constexpr int kMaxTeam = 18;
inline Partition make_partition(int B, int T, int out0, int kChunk, double handoff_cost, const std::vector<int>& dilations,
                                int grid, int force_G) {
  const int NC = (T - out0 + kChunk - 1) / kChunk;
  const int L = (int)dilations.size();
  std::vector<int> rsuf(L + 1, 0);
  for (int l = L - 1; l >= 0; l--) rsuf[l] = rsuf[l + 1] + dilations[l];
  const int warm_chunks = (rsuf[0] + kChunk - 1) / kChunk;
  std::vector<double> warm_cost(warm_chunks + 1, 0.0);
  for (int k = 0; k < warm_chunks; k++) {                      // chunk k ends k * kChunk rows before the first output row
    int lc = 0;
    while (lc < L && rsuf[lc + 1] > k * kChunk) lc++;
    warm_cost[k + 1] = warm_cost[k] + 0.1 + 0.9 * std::max(lc, 1) / (double)L;    // measured: flat optimum around (0.1, 0.9) .. (0, 1)
  }
  const long long total = (long long)B * NC;
  const int max_G = std::min(kMaxTeam, grid);
  auto teams_of = [&](int G) { return (int)std::min<long long>(grid / G, total); };
  auto fits = [&](int G) { return (long long)teams_of(G) * kMaxSeg >= B; };
  int only_G = 0;                                              // the forced size, lowered until it fits
  if (force_G > 0) {
    only_G = std::min(force_G, max_G);
    while (only_G > 1 && !fits(only_G)) only_G--;
  }
  Partition best;
  double best_time = 1e300;
  for (int G = 1; G <= max_G; G++) {
    if (only_G > 0 && G != only_G) continue;
    const int teams = teams_of(G);
    if (teams < 1 || !fits(G)) continue;
    Partition cand = partition_for(B, T, out0, kChunk, warm_cost, teams);
    if (cand.teams == 0) continue;
    const double lag = kLagLayers / L;
    const double period = std::max(1.0, G * lag);
    // measured (profiles/r02d_handoff_variants.log, r02e_team_sizes.log): a teacher chunk costs about 10 % more with the
    // hand-off (flag waits of the loader, row counting) than without; a student chunk about 4 % since its weight stage is
    // released by a plain arrive (32x64000: 1.825 ms with one CTA per piece, 1.725 ms with teams of 4)
    const double time = (cand.cost / G + (G > 1 ? 0.5 : 0.0)) * period * (G > 1 ? handoff_cost : 1.0) + (G - 1) * lag;
    if (time < best_time) { best_time = time; best = cand; best.G = G; }
  }
  return best;
}

}  // namespace fused
