"""The work partition of the fused kernel (csrc/partition.h), on the CPU: a small C++ driver built against the header
runs make_partition over batch sizes, lengths, stream offsets, forced team sizes, chunk lengths, SM counts and dilation
schedules.  Each partition must be one k_fused can run: every output row of every utterance exactly once, no team with
more than kMaxSeg pieces or more CTAs than the grid has, and enough warm-up before each piece's first output row for the
dependency cone of the layer stack.  The driver runs under a timeout, so a partition search that does not terminate
fails the test instead of hanging the suite."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from sr_wavenet_b200 import synth

CSRC = os.path.join(ROOT, "sr-wavenet_b200", "csrc")
K_MAX_SEG = 8
TEACHER = (384, 1.10)        # (rows per chunk, hand-off cost) as fused.cu's prepare() passes them
STUDENT = (512, 1.04)

DRIVER = r"""
#include "partition.h"
#include <cstdio>
#include <vector>
// stdin: one case per line: B T out0 chunk handoff grid force_G L d_0 .. d_{L-1}
// stdout per case: "teams G", then per team: nseg followed by b t_start t_out t_end of each segment
int main() {
  int B, T, out0, chunk, grid, force_G, L;
  double handoff;
  while (scanf("%d %d %d %d %lf %d %d %d", &B, &T, &out0, &chunk, &handoff, &grid, &force_G, &L) == 8) {
    std::vector<int> dil(L);
    for (int& d : dil) if (scanf("%d", &d) != 1) return 2;
    const fused::Partition p = fused::make_partition(B, T, out0, chunk, handoff, dil, grid, force_G);
    printf("%d %d\n", p.teams, p.G);
    for (int tm = 0; tm < p.teams; tm++) {
      printf("%d", p.nseg[tm]);
      for (int i = 0; i < p.nseg[tm]; i++) {
        const fused::Seg& s = p.segs[(size_t)tm * fused::kMaxSeg + i];
        printf(" %d %d %d %d", s.b, s.t_start, s.t_out, s.t_end);
      }
      printf("\n");
    }
    fflush(stdout);
  }
  return 0;
}
"""

DEFAULT = list(synth.DEFAULT_DILATIONS)
DILATIONS = {"default": DEFAULT, "1_512": [1, 512], "40_layers": [1 << (i % 10) for i in range(40)]}


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    d = tmp_path_factory.mktemp("partition")
    src, exe = d / "driver.cpp", d / "driver"
    src.write_text(DRIVER)
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", CSRC, str(src), "-o", str(exe)],
                   check=True)
    return str(exe)


def run(driver, cases, timeout=60):
    """cases: (B, T, out0, (chunk, handoff), grid, force_G, dilations) -> [(teams, G, [[(b, t_start, t_out, t_end)]])]"""
    lines = ["%d %d %d %d %.17g %d %d %d %s" % (B, T, out0, kind[0], kind[1], grid, g, len(dil), " ".join(map(str, dil)))
             for B, T, out0, kind, grid, g, dil in cases]
    try:
        out = subprocess.run([driver], input="\n".join(lines) + "\n", capture_output=True, text=True, timeout=timeout,
                             check=True).stdout.split("\n")
    except subprocess.TimeoutExpired:
        pytest.fail("the partition search did not terminate within %d s" % timeout)
    res, i = [], 0
    for _ in cases:
        teams, G = map(int, out[i].split())
        i += 1
        pieces = []
        for _ in range(teams):
            v = list(map(int, out[i].split()))
            i += 1
            pieces.append([tuple(v[1 + 4 * k:5 + 4 * k]) for k in range(v[0])])
        res.append((teams, G, pieces))
    return res


def history(dil):
    """The stream call's carried rows: the flow's dependency window sum(d) + 2, rounded up to pool_stride 128."""
    return (sum(dil) + 2 + 127) // 128 * 128


def check(case, teams, G, pieces):
    B, T, out0, (chunk, _), grid, force_G, dil = case
    assert teams >= 1 and G >= 1, case
    assert teams * G <= grid, case
    assert len(pieces) == teams
    if force_G:                                                # kept if its grid / G teams hold B, else lowered
        Gf = min(force_G, 18, grid)
        total = B * -(-(T - out0) // chunk)
        assert G == Gf if min(grid // Gf, total) * K_MAX_SEG >= B else G < Gf, case
    need = sum(dil)
    segs = np.array([s for p in pieces for s in p], dtype=np.int64).reshape(-1, 4)
    for p in pieces:
        assert len(p) <= K_MAX_SEG, case          # a team may be idle (few long utterances, large forced G)
    b, ts, to, te = segs.T
    assert ((b >= 0) & (b < B)).all(), case
    assert ((ts <= to) & (to < te) & (te <= T)).all(), case
    # a piece that starts mid-utterance rebuilds every layer's history: h_0 is exact from t_start on (the front conv reads
    # x itself, zero before row 0), and the stack reaches sum(d) rows back, so t_out - t_start >= sum(d) unless the
    # piece starts at row 0, where the zero padding before it is the utterance's own
    assert ((to - ts >= np.minimum(to, need)) | (ts == 0)).all(), case
    assert ((ts == 0) | (to - ts >= need)).all(), case
    # per utterance: [t_out, t_end) ranges tile [out0, T) exactly once, in order, and the first piece starts at row 0
    order = np.lexsort((to, b))
    b, ts, to, te = b[order], ts[order], to[order], te[order]
    assert np.array_equal(np.unique(b), np.arange(B)), case
    first = np.r_[True, b[1:] != b[:-1]]
    last = np.r_[b[1:] != b[:-1], True]
    assert (to[first] == out0).all() and (ts[first] == 0).all(), case
    assert (te[last] == T).all(), case
    assert (to[~first] == te[np.nonzero(~first)[0] - 1]).all(), case
    # output pieces start on chunk boundaries counted from out0 (the kernel's warm/head decision is per chunk)
    assert ((to - out0) % chunk == 0).all(), case


BATCHES = [1, 2, 63, 64, 65, 148, 149, 500, 1184]


def lengths(B, chunk):
    """One chunk, a few chunks with a ragged tail, past the receptive field, and 64000 where the batch keeps it cheap."""
    Ts = [chunk, 3 * chunk + 128, 4096 + 128 * 3]
    if B <= 149:
        Ts.append(64000)
    return Ts


def cases_for(B):
    out = []
    for name, dil in DILATIONS.items():
        for kind in (TEACHER, STUDENT):
            for T in lengths(B, kind[0]):
                for out0 in (0, history(dil)):
                    for grid in (148, 132):
                        for g in (0, 1, 2, 7, 18):
                            out.append((B, T + out0, out0, kind, grid, g, dil))
    return out


@pytest.mark.parametrize("B", BATCHES)
def test_partition_covers_every_output_row_once(driver, B):
    cases = cases_for(B)
    feasible = [c for c in cases if c[0] <= c[4] * K_MAX_SEG]
    for case, (teams, G, pieces) in zip(feasible, run(driver, feasible)):
        check(case, teams, G, pieces)


def test_forced_team_size_is_lowered_until_the_batch_fits(driver):
    """148 SMs / 18 = 8 teams hold 64 utterances: a forced size of 18 stays at 65 only if lowered (to 16: 9 teams)."""
    (t64, g64, _), (t65, g65, _), (t1184, g1184, _) = run(driver, [
        (64, 384, 0, TEACHER, 148, 18, DEFAULT), (65, 384, 0, TEACHER, 148, 18, DEFAULT),
        (1184, 384, 0, TEACHER, 148, 18, DEFAULT)])
    assert (t64, g64) == (8, 18)
    assert (t65, g65) == (9, 16)
    assert (t1184, g1184) == (148, 1)


def test_batch_past_the_segment_limit_is_infeasible(driver):
    """148 SMs x kMaxSeg = 1184 utterances: one more has no partition, whatever the team size (the library refuses it
    before any launch)."""
    res = run(driver, [(1185, 384, 0, TEACHER, 148, 1, DEFAULT), (1185, 384, 0, TEACHER, 148, 0, DEFAULT),
                       (1185, 512, 0, STUDENT, 148, 0, DEFAULT), (1057, 512, 0, STUDENT, 132, 0, DEFAULT),
                       (1184, 384, 0, TEACHER, 148, 1, DEFAULT)])
    assert [r[:2] for r in res[:4]] == [(0, 0)] * 4
    assert res[4][:2] == (148, 1)


def test_bench_shapes_keep_their_partitions(driver):
    """The partitions of the benchmark shapes (default 30 layers on 148 SMs), measured as chosen before the search was
    bounded: the bound must not move them."""
    res = run(driver, [(32, 64000, 0, TEACHER, 148, 0, DEFAULT), (4, 64000, 0, TEACHER, 148, 0, DEFAULT),
                       (1, 64000, 0, TEACHER, 148, 0, DEFAULT), (8, 64000, 0, STUDENT, 148, 0, DEFAULT)])
    assert [r[:2] for r in res] == [(148, 1), (12, 12), (11, 13), (16, 9)]
