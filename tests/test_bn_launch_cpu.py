"""Launch geometry of the BatchNorm passes (abcnet_b200/csrc/bn_launch.cuh), checked on the CPU: a host-only probe compiled
with nvcc prints bn_launch_config for a spread of shapes on a 148-SM B200. The expected grids are the ones the launchers of
abc_bn_stats / abc_channel_sum (stats), abc_bn_act, abc_bn_act_backward and abc_nchw_to_p8_ex (pixels, or pool with a fused
2x2 max-pool) computed before they shared the helper."""
import os
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abcnet_b200", "csrc")

# (N, planes, H, W) -> grid.x of the stats, pixels and pool passes (None: odd H or W, no pooled pass).
# planes = 1 stands for C = 8, and for C = 1 in abc_nchw_to_p8_ex.
GRID_X = [
    ((1, 1, 1, 1), (1, 1, None)),
    ((1, 1, 2, 2), (1, 1, 1)),
    ((3, 4, 7, 5), (1, 1, None)),
    ((1, 1, 1, 4096), (4, 8, None)),
    ((1, 1, 512, 512), (256, 512, 256)),
    ((1, 1, 2048, 2048), (1776, 1776, 1776)),
    ((2, 4, 100, 64), (7, 13, 7)),
    ((8, 2, 96, 96), (9, 18, 9)),
    ((64, 2, 64, 64), (4, 8, 4)),
    ((64, 2, 512, 512), (14, 14, 14)),
    ((64, 4, 256, 256), (7, 7, 7)),
    ((64, 8, 128, 128), (4, 4, 4)),
    ((64, 16, 64, 64), (2, 2, 2)),
    ((64, 128, 128, 128), (1, 1, 1)),
    ((256, 16, 32, 32), (1, 1, 1)),
    ((60000, 2, 4, 4), (1, 1, 1)),
]
PASSES = ("kStats", "kPixels", "kPool")


def test_bn_launch_config_matches_previous_grids(tmp_path):
    lines = ['#include <cstdio>', '#include "bn_launch.cuh"', "using namespace abc;", "int main() {"]
    cases = []
    for (N, P, H, W), xs in GRID_X:
        for name, x in zip(PASSES, xs):
            if x is None:
                continue
            cases.append(((N, P, H, W), name, x))
            lines.append(f"  {{ const BnLaunch l = bn_launch_config(BnPass::{name}, {N}, {P}, {H}, {W}, 148);"
                         ' printf("%u %u %u %d\\n", l.grid.x, l.grid.y, l.grid.z, l.block); }')
    lines += ["  return 0;", "}"]
    src = tmp_path / "probe.cu"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.run([nvcc, "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], check=True)
    env = {k: v for k, v in os.environ.items() if k != "ABCNET_BN_BLOCKS_PER_SM"}
    got = subprocess.run([str(exe)], capture_output=True, text=True, check=True, env=env).stdout.splitlines()
    assert len(got) == len(cases)
    for ((N, P, H, W), name, x), line in zip(cases, got):
        assert tuple(map(int, line.split())) == (x, P, N, 256), f"{name} N={N} planes={P} H={H} W={W}: {line}"
