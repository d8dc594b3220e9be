"""Host-side logic that needs no GPU: the SYRK's work decomposition (csrc/oz8.cu: O8SegIter, shared by the kernel's warp roles,
the finishing kernel and the host sizing code) compiled for the CPU and checked exhaustively, and the C demo of the whole-step
entry points compiled and linked against include/npgp.h + libnpgp.so with a plain C compiler."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = r"""
#include <cstdio>
#include <map>
#include <vector>
constexpr int O8_MAX_SEG = 512;
%s
int main() {
  int cases[][3] = {{72, 2048, 228}, {72, 256, 86}, {72, 4, 4}, {272, 2048, 512}, {3, 7, 7}, {72, 2047, 228}, {8, 3000, 500},
                    {1, 1, 1}, {148, 33, 32}, {149, 64, 64}};
  int bad_total = 0;
  for (auto& cs : cases) {
    const int nt = cs[0], nks = cs[1], spc = cs[2];
    const long items = (long)nt * ((nks + spc - 1) / spc);
    const int G = (int)(items < 148 ? items : 148);
    std::vector<int> cov((long)nt * nks, 0);
    std::map<long, std::vector<std::pair<int, int>>> segs;
    long mx = 0;
    int bad = 0;
    for (int c = 0; c < G; ++c) {
      O8SegIter it(nt, nks, spc, c, G);
      int t, k0, k1, cnt = 0;
      long st = 0;
      while (it.next(t, k0, k1)) {
        if (k1 - k0 > O8_MAX_SEG || k1 <= k0 || k1 > nks || k0 / spc != (k1 - 1) / spc || t < 0 || t >= nt) ++bad;
        for (int k = k0; k < k1; ++k) cov[(long)t * nks + k]++;
        segs[(long)t * 100000 + k0 / spc].push_back({c, cnt});
        ++cnt;
        st += k1 - k0;
      }
      if (st > mx) mx = st;
    }
    for (auto v : cov) bad += v != 1;  // every (tile, stage) exactly once
    // the finishing kernel's enumeration finds exactly the segments the CTAs produced, in the same order
    O8SegIter probe(nt, nks, spc, 0, G);
    const long LB = probe.remainder_share();
    const int nch = (nks + spc - 1) / spc;
    for (int tile = 0; tile < nt; ++tile)
      for (int ch = 0; ch < nch; ++ch) {
        const int item = ch * nt + tile;
        std::vector<std::pair<int, int>> got;
        if (item < probe.full * G) got.push_back({item %% G, item / G});
        else {
          const int j = item - probe.full * G;
          const int cf = (int)(((long)j * spc) / LB), cl = (int)((((long)j + 1) * spc - 1) / LB);
          for (int c = cf; c <= cl && c < G; ++c) {
            O8SegIter it(nt, nks, spc, c, G, true);
            int t2, k0, k1, idx = probe.full;
            while (it.next(t2, k0, k1)) {
              if (t2 == tile && k0 / spc == ch) got.push_back({c, idx});
              ++idx;
            }
          }
        }
        bad += got != segs[(long)tile * 100000 + ch];
      }
    const double ideal = (double)nt * nks / G;
    // balanced: with the remainder split no CTA runs more than ideal + one chunk-rounding's worth of stages
    if (mx > ideal + spc + 1) ++bad;
    printf("nt=%%d nks=%%d spc=%%d G=%%d bad=%%d max=%%ld ideal=%%.1f\n", nt, nks, spc, G, bad, mx, ideal);
    bad_total += bad;
  }
  return bad_total ? 1 : 0;
}
"""


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs a host C++ compiler")
def test_syrk_segment_iterator_covers_every_stage_once_and_finish_agrees(tmp_path):
    src = open(os.path.join(ROOT, "nonstationary_precip_b200", "csrc", "oz8.cu")).read()
    m = re.search(r"struct O8SegIter \{.*?\n\};", src, re.S)
    assert m, "O8SegIter not found in oz8.cu"
    body = m.group(0).replace("__host__ __device__", "")
    cpp = tmp_path / "segiter.cpp"
    cpp.write_text(HARNESS % body)
    exe = str(tmp_path / "segiter")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", exe, str(cpp)], check=True, capture_output=True, text=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.skipif(shutil.which("gcc") is None or not os.path.exists("/usr/local/cuda/include/cuda_runtime.h"),
                    reason="needs gcc and the CUDA headers")
def test_c_demo_compiles_and_links_against_the_header(tmp_path):
    """include/npgp.h is plain C and libnpgp.so exports what the whole-step demo calls (no GPU needed to link)."""
    libdir = os.path.join(ROOT, "nonstationary_precip_b200")
    if not os.path.exists(os.path.join(libdir, "libnpgp.so")):
        pytest.skip("libnpgp.so not built")
    exe = str(tmp_path / "svgp_step_demo")
    cmd = ["gcc", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
           os.path.join(ROOT, "tools", "c_demo", "svgp_step_demo.c"), "-o", exe, "-L", libdir, "-lnpgp",
           "-L", "/usr/local/cuda/lib64", "-lcudart", "-lm", "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert os.path.exists(exe)
