"""Slot arithmetic of the deterministic reductions (abcnet_b200/csrc/det_slots.cuh), checked on the CPU: a host-only probe
compiled with nvcc prints slot counts and workspace bytes for the layers of the v2 network at B = 64, 512 x 512 and for edge
shapes; the expected values follow the launch geometry of abc_conv_wgrad (split-K grid.x) and bn_launch_config on a
148-SM B200."""
import os
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abcnet_b200", "csrc")
SMS = 148

# wgrad of the v2 training step at B = 64, 512 x 512: (cout, cin, H, W, ntaps) + edge shapes (partial tiles, 1 x 1 images)
WGRAD = [(16, 16, 512, 512, 9), (32, 16, 256, 256, 9), (32, 32, 256, 256, 9), (64, 32, 128, 128, 9), (64, 64, 128, 128, 9),
         (128, 64, 64, 64, 9), (128, 128, 64, 64, 9), (256, 128, 32, 32, 9), (256, 256, 32, 32, 9), (512, 256, 16, 16, 9),
         (512, 512, 16, 16, 9), (1024, 128, 128, 128, 9), (16, 128, 128, 128, 1), (368, 128, 128, 128, 1), (256, 512, 16, 16, 4),
         (8, 16, 1, 1, 9), (24, 16, 17, 9, 9), (8, 16, 1, 1, 1)]


def wgrad_grid(cout, cin, H, W, ntaps, N):
    """grid of abc_conv_wgrad (wgrad_sm100.cu): n_tile = min(cin, 128), taps per CTA from the 512 TMEM columns."""
    n_tile = cin if cin < 128 else 128
    tpc = min(512 // n_tile, ntaps)
    if ntaps == 9 and tpc < 9:
        tpc = 3 if tpc >= 3 else 1
    if ntaps == 4 and tpc < 4:
        tpc = 2 if tpc >= 2 else 1
    gy = ((cout + 127) // 128) * (cin // n_tile) * ((ntaps + tpc - 1) // tpc)
    tiles = N * ((W + 7) // 8) * ((H + 15) // 16)
    return min(max(SMS // gy, 1), tiles), gy


def bn_grid_x(N, planes, H, W, per_thread):
    items, per_block = H * W, 256 * per_thread
    need, cap = (items + per_block - 1) // per_block, (SMS * 12 + planes * N - 1) // (planes * N)
    return max(1, min(need, cap))


BN = [(64, 2, 512, 512), (64, 4, 256, 256), (64, 8, 128, 128), (64, 16, 64, 64), (64, 32, 32, 32), (64, 64, 16, 16),
      (64, 128, 128, 128), (1, 1, 1, 1), (3, 3, 7, 5), (64, 46, 128, 128)]


def test_slot_counts_and_workspace_bytes(tmp_path):
    lines = ['#include <cstdio>', '#include "det_slots.cuh"', "using namespace abc;", "int main() {"]
    for cout, cin, H, W, ntaps in WGRAD:
        N = 64
        gy = wgrad_grid(cout, cin, H, W, ntaps, N)[1]
        tiles = N * ((W + 7) // 8) * ((H + 15) // 16)
        lines.append(f'  {{ const int gx = wgrad_grid_x({SMS}, {gy}, {tiles});'
                     f' printf("%d %zu\\n", gx, det_ws_bytes(gx, {ntaps * cout * cin}ll, 4)); }}')
    for N, P, H, W in BN:
        for name in ("kStats", "kPixels", "kPool"):
            lines.append(f'  {{ const BnLaunch l = bn_launch_config(BnPass::{name}, {N}, {P}, {H}, {W}, {SMS});'
                         f' printf("%d %zu %d\\n", bn_slots(l), det_ws_bytes(bn_slots(l), {16 * P}ll, 8), bn_slot(1, 2, l.grid.x)); }}')
    lines.append('  printf("%zu %d %d %d\\n", det_slot_index(3, 7, 2), conv_stat_slots(18), loss_elems(false, 60), loss_elems(true, 60));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "probe.cu"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.run([nvcc, "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], check=True)
    env = {k: v for k, v in os.environ.items() if k != "ABCNET_BN_BLOCKS_PER_SM"}
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True, env=env).stdout.splitlines()
    it = iter(out)
    for cout, cin, H, W, ntaps in WGRAD:
        gx, gy = wgrad_grid(cout, cin, H, W, ntaps, 64)
        got = tuple(map(int, next(it).split()))
        assert got == (gx, gx * ntaps * cout * cin * 4), (cout, cin, H, W, ntaps, got)
        # every split-K CTA of a column writes one [128 x <= 512] TMEM block: the workspace never exceeds max(SMs, gy) of them
        assert got[1] <= max(SMS, gy) * 128 * 512 * 4
    for N, P, H, W in BN:
        for per_thread, pooled in ((4, False), (2, False), (1, True)):
            hh, ww = (H // 2, W // 2) if pooled else (H, W)
            gx = bn_grid_x(N, P, hh, ww, per_thread)
            got = tuple(map(int, next(it).split()))
            assert got == (gx * N, gx * N * 16 * P * 8, 2 * gx + 1), (N, P, H, W, per_thread, got)
    assert tuple(map(int, next(it).split())) == (23, 144, 16, 16 + 2 + 19 + 480)
