"""How abc_heads_fused splits its persistent CTAs among the head pairs (abcnet_b200/csrc/heads_split.cuh), checked on the
CPU: a host-only probe compiled with nvcc prints the per-pair tile costs and CTA counts for several head lists."""
import itertools
import os
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abcnet_b200", "csrc")

V2_HEADS = [1, 14, 3, 2, 1, 360, 60, 60]


def _chunks(pair):
    """conv2 chunk widths of a head pair, as abc_heads_fused builds them: <= 128 channels each, rounded up to 16."""
    return [(min(h - c0, 128) + 15) // 16 * 16 for h in pair for c0 in range(0, h, 128)]


def _probe(tmp_path, cases):
    """cases: (heads, sms, num_tiles) -> per case (costs, ctas, total) from the C++ helpers."""
    lines = ['#include <cstdio>', '#include "heads_split.cuh"', "using namespace abc;", "int main() {"]
    for heads, sms, tiles in cases:
        pairs = [heads[i:i + 2] for i in range(0, len(heads), 2)]
        lines.append("  {")
        lines.append(f"    int64_t cost[{len(pairs)}]; int ctas[{len(pairs)}];")
        for k, pr in enumerate(pairs):
            nc = _chunks(pr)
            lines.append(f"    {{ const int nc[] = {{{', '.join(map(str, nc))}}}; cost[{k}] = hf_pair_tile_cost({len(nc)}, nc, {sum(pr)}); }}")
        lines.append(f"    const int total = hf_split_ctas({len(pairs)}, cost, {sms}, {tiles}, ctas);")
        lines.append(f'    printf("%d", total); for (int i = 0; i < {len(pairs)}; ++i) printf(" %lld %d", (long long)cost[i], ctas[i]); printf("\\n");')
        lines.append("  }")
    lines += ["  return 0;", "}"]
    src = tmp_path / "probe.cu"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.run([nvcc, "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], check=True)
    out = []
    for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines():
        v = list(map(int, line.split()))
        out.append((v[1::2], v[2::2], v[0]))
    return out


def _max_share(cost, ctas):
    return max(c / n for c, n in zip(cost, ctas))


def test_pair_split_follows_the_cost_per_tile(tmp_path):
    cases = [(V2_HEADS, 148, 32768), ([1, 21, 5, 1, 4, 2], 148, 4096), ([1, 14, 3], 148, 96), ([360], 148, 32768),
             (V2_HEADS, 20, 32768), (V2_HEADS, 3, 32768), (V2_HEADS, 148, 10), ([1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16], 148, 1000)]
    for (heads, sms, tiles), (cost, ctas, total) in zip(cases, _probe(tmp_path, cases)):
        pairs = [heads[i:i + 2] for i in range(0, len(heads), 2)]
        assert len(ctas) == len(pairs) and total == sum(ctas)
        assert all(n >= 1 for n in ctas)
        assert all(n <= max(1, tiles) for n in ctas)
        # every SM is used unless each pair already has a CTA per tile, and never more CTAs than SMs unless a pair would get none
        assert total == min(max(sms, len(pairs)), len(pairs) * tiles)
        # the cost model grows with the conv2 chunks and the logit channels of the pair
        for i, j in itertools.permutations(range(len(pairs)), 2):
            if sorted(_chunks(pairs[i])) == sorted(_chunks(pairs[j])) and sum(pairs[i]) == sum(pairs[j]):
                assert cost[i] == cost[j]
            if sum(_chunks(pairs[i])) > sum(_chunks(pairs[j])) and sum(pairs[i]) > sum(pairs[j]) and len(_chunks(pairs[i])) >= len(_chunks(pairs[j])):
                assert cost[i] > cost[j]
        # no single CTA moved from one pair to another lowers the largest cost per CTA (the greedy split is optimal)
        best = _max_share(cost, ctas)
        for i, j in itertools.permutations(range(len(pairs)), 2):
            if ctas[i] > 1 and ctas[j] < tiles:
                moved = list(ctas)
                moved[i] -= 1
                moved[j] += 1
                assert _max_share(cost, moved) >= best
    # the v2 heads on a B200: the 1 + 360-channel pair gets the most CTAs, the two light pairs the fewest
    cost, ctas, _ = _probe(tmp_path, [(V2_HEADS, 148, 32768)])[0]
    assert ctas[2] == max(ctas) and ctas[2] > 37 and min(ctas) in (ctas[0], ctas[1])
