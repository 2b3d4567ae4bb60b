"""The slot arithmetic of the sparse-heads path (abcnet_b200/csrc/peak_slots.cuh), checked on the CPU: a host-only probe
compiled with nvcc reads count vectors, runs the header's offsets / slot -> (group, index) / per-group slot counts in both
layouts, and prints them for comparison with numpy."""
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abcnet_b200", "csrc")

_PROBE = r"""
#include <cstdio>
#include <vector>
#include "peak_slots.cuh"
using namespace abc;
// stdin: cases of "groups pool cap runs cnt[0..groups)"; pool > 0 selects the pooled layout, cap > 0 the fixed one.
// stdout per case: offsets (pooled: groups + 1 values, computed in `runs` consecutive pieces as the device kernel does),
// then slot_count per group, then for every slot "g i" (i = -1 when the slot holds no peak).
int main() {
  int G, pool, cap, runs;
  while (std::scanf("%d %d %d %d", &G, &pool, &cap, &runs) == 4) {
    std::vector<int32_t> cnt(G), off(G + 1, -7);
    for (int g = 0; g < G; ++g) std::scanf("%d", &cnt[g]);
    SlotLayout L{nullptr, cap, pool, cap};
    int P = G * cap;
    if (pool > 0) {
      const int per = (G + runs - 1) / runs;
      int base = 0;
      for (int r = 0; r < runs; ++r) {
        const int b0 = r * per < G ? r * per : G, b1 = b0 + per < G ? b0 + per : G;
        base = slot_offsets(cnt.data() + b0, b1 - b0, base, off.data() + b0);
      }
      off[G] = base;
      L = SlotLayout{off.data(), 0, pool, 1 << 14};
      P = pool;
      for (int g = 0; g <= G; ++g) std::printf("%d ", off[g]);
    }
    std::printf("\n");
    for (int g = 0; g < G; ++g) std::printf("%d ", slot_count(L, g, cnt[g]));
    std::printf("\n");
    for (int s = 0; s < P; ++s) {
      const int g = slot_group(L, s, G), i = s - slot_base(L, g);
      std::printf("%d %d ", g, i < slot_count(L, g, cnt[g]) ? i : -1);
    }
    std::printf("\n");
  }
  return 0;
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    d = tmp_path_factory.mktemp("peak_slots")
    src, exe = d / "probe.cu", d / "probe"
    src.write_text(_PROBE)
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.run([nvcc, "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], check=True)

    def run(cases):
        text = "".join(f"{len(c)} {pool} {cap} {runs} {' '.join(map(str, c))}\n" for c, pool, cap, runs in cases)
        lines = subprocess.run([str(exe)], input=text, capture_output=True, text=True, check=True).stdout.split("\n")
        out = []
        for k, (c, pool, cap, runs) in enumerate(cases):
            off, scount, pairs = (np.array(lines[3 * k + j].split(), dtype=np.int64) for j in range(3))
            out.append((off, scount, pairs.reshape(-1, 2)))
        return out
    return run


def _expected_pooled(cnt, pool):
    """numpy model of the pooled layout: slot s belongs to the peak whose running index over the groups is s, if s < pool."""
    off = np.concatenate([[0], np.cumsum(cnt)])
    scount = np.clip(np.minimum(cnt, pool - off[:-1]), 0, None)
    pairs = np.full((pool, 2), -1, np.int64)
    for g, c in enumerate(cnt):
        for i in range(c):
            if off[g] + i < pool:
                pairs[off[g] + i] = (g, i)
    return off, scount, pairs


def test_pooled_offsets_and_inverse(probe):
    rng = np.random.default_rng(5)
    S = 512
    cases = [np.zeros(8, np.int64),                                       # no peaks at all
             np.array([0, 0, S, 0, 0, 0]),                                # one image holds the whole pool
             np.array([S - 40, 0, 0, 40]),                                # exact fit, empty groups in between
             np.array([0, 0, 0, 0, 0, S]),                                # the last group fills it
             np.array([5, 0, 0, 3, 0, 0, 0, 2]),                          # runs of empty groups
             np.array([300, 300, 10, 1]),                                 # overflow inside group 1
             np.array([S + 1]),                                           # one group, one peak too many
             np.array([S, 7, 0, 9])]                                      # overflow right at a group boundary
    cases += [rng.integers(0, 60, size=int(rng.integers(1, 70))) * (rng.random() < 0.8) for _ in range(40)]
    cases += [np.where(rng.random(2 * 37) < 0.7, 0, rng.integers(0, 200, 2 * 37)) for _ in range(10)]
    runs = [1, 3, 1024]
    got = probe([(list(map(int, c)), S, 0, runs[k % 3]) for k, c in enumerate(cases)])
    for c, (off, scount, pairs) in zip(cases, got):
        want_off, want_count, want_pairs = _expected_pooled(np.asarray(c, np.int64), S)
        assert np.array_equal(off, want_off), (c, off)
        assert np.array_equal(scount, want_count), c
        valid = pairs[:, 1] >= 0
        assert np.array_equal(pairs[valid], want_pairs[want_pairs[:, 1] >= 0]), c
        assert np.array_equal(valid, want_pairs[:, 1] >= 0), c
        # the overflow rule: every peak has a slot exactly when the total fits the pool
        total = int(np.sum(c))
        assert int(scount.sum()) == min(total, S)
        assert (int(scount.sum()) < total) == (total > S)
        # slot -> (g, i) -> slot is the identity on the slots that hold a peak
        g, i = pairs[valid, 0], pairs[valid, 1]
        assert np.array_equal(want_off[g] + i, np.flatnonzero(valid))


def test_fixed_layout_is_g_times_cap(probe):
    cap = 64
    cases = [np.array([0, 64, 65, 3]), np.array([1000, 0]), np.array([64] * 6)]
    for c, (off, scount, pairs) in zip(cases, probe([(list(map(int, c)), 0, cap, 1) for c in cases])):
        assert off.size == 0
        assert np.array_equal(scount, np.minimum(c, cap))                 # truncated at peak_cap
        s = np.arange(len(c) * cap)
        assert np.array_equal(pairs[:, 0], s // cap)
        assert np.array_equal(pairs[:, 1], np.where(s % cap < np.minimum(c, cap)[s // cap], s % cap, -1))
