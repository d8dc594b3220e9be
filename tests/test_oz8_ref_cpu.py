"""The exact reference of the int8 digit contractions (tests/oz8_ref.py) checked without a GPU: plane layouts round-trip,
the GEMM-based digit products and their recombination agree with Python integer arithmetic, and the port of the SYRK's
work split (O8SegIter, o8_syrk_shape of csrc/oz8.cu) agrees with the C++ compiled from the source itself."""
import math
import os
import re
import shutil
import subprocess
import sys
from fractions import Fraction

import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))
import oz8_ref as R  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plane_layouts_round_trip():
    g = torch.Generator().manual_seed(1)
    D = torch.randint(-128, 128, (7, 256, 96), generator=g, dtype=torch.int8)
    assert torch.equal(R.a_digits(R.encode_a_planes(D), 256, 96), D)
    assert torch.equal(R.decode_planes(R.encode_a_planes(D), 256, 96), R.digits_value(D).double())
    Db = torch.randint(-128, 128, (7, 192, 64), generator=g, dtype=torch.int8)
    assert torch.equal(R.b_digits(R.encode_b_planes(Db), 192, 64), Db)


def python_reference(a, b):
    """One output entry from two digit rows a, b (lists of 7 lists of ints) in Python integers: G_t, hi, lo, and the
    recombined double fma(lo, 2^-24, hi) = float(hi) + float(lo) 2^-24 with Python's correctly rounded conversions."""
    K = len(a[0])
    G = [sum(a[p][k] * b[t - p][k] for p in range(t + 1) for k in range(K)) for t in range(7)]
    hi = ((G[0] * 256 + G[1]) * 256 + G[2]) * 256 + G[3]
    lo = (G[4] * 256 + G[5]) * 256 + G[6]
    return G, hi, lo, float(hi) + float(lo) * 2.0 ** -24


@pytest.mark.parametrize("kind", ["random", "min", "max", "mixed"])
def test_gemm_reference_agrees_with_python_integers(kind):
    g = torch.Generator().manual_seed(len(kind))
    n, N, Kd = 3, 4, 2048
    if kind == "random":
        DA = torch.randint(-128, 128, (7, n, Kd), generator=g, dtype=torch.int8)
        DB = torch.randint(-128, 128, (7, N, Kd), generator=g, dtype=torch.int8)
    else:
        va, vb = {"min": (-128, -128), "max": (127, 127), "mixed": (-128, 127)}[kind]
        DA, DB = torch.full((7, n, Kd), va, dtype=torch.int8), torch.full((7, N, Kd), vb, dtype=torch.int8)
    ea = torch.tensor([-960, 0, 700], dtype=torch.int32)
    eb = torch.tensor([5, -3, 0, R.POISON], dtype=torch.int32)
    G = R.digit_products(DA, DB)
    T = R.gemm_reference(DA, ea, DB, eb, row_block=2)
    for i in range(n):
        for j in range(N):
            Gp, hi, lo, v = python_reference(DA[:, i].tolist(), DB[:, j].tolist())
            assert G[:, i, j].long().tolist() == Gp
            assert R.recombine(G[:, i:i + 1, j:j + 1]).item() == v
            if abs(hi) < 2 ** 53:  # then the recombination is the correctly rounded exact sum
                assert v == float(Fraction(hi) + Fraction(lo, 2 ** 24))
            if eb[j] == R.POISON:
                assert math.isnan(T[i, j].item())
            else:
                want = v * 2.0 ** (int(ea[i]) - 36) * 2.0 ** int(eb[j])
                assert T[i, j].item() == want


def test_pow2_and_exponents():
    k = torch.arange(-1022, 1024)
    assert torch.equal(R.pow2(k), torch.tensor([math.ldexp(1.0, int(v)) for v in k], dtype=torch.float64))
    assert R.exponent_of_scale(0.644) == 0 and R.exponent_of_scale(1.0) == 1 and R.exponent_of_scale(2.0 ** -2000) == R.POISON
    assert R.exponent_of_scale(1e-300) == R.EMIN


HARNESS = r"""
#include <cstdio>
constexpr int O8_MAX_SEG = 512;
constexpr int O8_KS = 32;
constexpr int O8_NS = 7;
constexpr int kNumSMs = 148;
static inline int ceil_div(long a, long b) { return (int)((a + b - 1) / b); }
%s
%s
int main() {
  int nm[][2] = {%s};
  for (auto& c : nm) {
    const int n = c[0], M = c[1];
    const int nks = ceil_div(((long)n + 127) / 128 * 128, 32);
    const int n_rb = M / 128, n_cb = M / 64, nt = n_rb * n_cb - n_rb * (n_rb - 1);
    int G, spc;
    const int slots = o8_syrk_shape(nks, nt, M, &G, &spc);
    printf("shape %%d %%d %%d %%d %%d\n", n, M, G, spc, slots);
    for (int cta = 0; cta < G; ++cta) {
      O8SegIter it(nt, nks, spc, cta, G);
      int t, k0, k1;
      while (it.next(t, k0, k1)) printf("seg %%d %%d %%d %%d %%d\n", cta, t, k0, k1, 0);
    }
  }
  return 0;
}
"""

CASES = [(4100, 1024), (1, 128), (119168, 128), (30000, 1024), (21760, 1024), (120832, 128), (65536, 1024), (16384, 4096),
         (16512, 4096), (20000, 512), (30000, 256), (777, 384)]


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs a host C++ compiler")
def test_work_split_port_matches_the_compiled_source(tmp_path):
    src = open(os.path.join(ROOT, "nonstationary_precip_b200", "csrc", "oz8.cu")).read()
    it = re.search(r"struct O8SegIter \{.*?\n\};", src, re.S)
    shape = re.search(r"static int o8_syrk_shape\(.*?\n\}", src, re.S)
    assert it and shape, "O8SegIter / o8_syrk_shape not found in oz8.cu"
    cpp = tmp_path / "split.cpp"
    cpp.write_text(HARNESS % (it.group(0).replace("__host__ __device__", ""), shape.group(0),
                              ", ".join("{%d, %d}" % c for c in CASES)))
    exe = str(tmp_path / "split")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", exe, str(cpp)], check=True, capture_output=True, text=True)
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split("\n")
    pos = 0
    for n, M in CASES:
        plan = R.syrk_plan(n, M)
        assert out[pos] == "shape %d %d %d %d %d" % (n, M, plan["n_cta"], plan["spc"], plan["slots"])
        pos += 1
        for c in range(plan["n_cta"]):
            for t, k0, k1 in R.cta_segments(plan["n_tiles"], plan["nks"], plan["spc"], c, plan["n_cta"]):
                assert out[pos] == "seg %d %d %d %d 0" % (c, t, k0, k1)
                pos += 1
    assert out[pos:] == [""]


@pytest.mark.parametrize("n,M", CASES)
def test_finish_order_is_the_segment_order_along_the_contraction(n, M):
    """The finishing kernel adds a tile's partials chunk by chunk and, inside a remainder item, CTA by CTA; each CTA's
    range is contiguous, so that order is ascending k0 with the segments tiling [0, nks) without gaps.  The reference adds
    them in exactly this order."""
    plan = R.syrk_plan(n, M)
    full, G, spc, nt = plan["full"], plan["n_cta"], plan["spc"], plan["n_tiles"]
    for tile, segs in enumerate(plan["segments"]):
        ks = [k for seg in segs for k in seg[:2]]
        assert ks[0] == 0 and ks[-1] == plan["nks"] and all(ks[2 * i + 1] == ks[2 * i + 2] for i in range(len(segs) - 1))
        for k0, k1, c, idx in segs:
            item = (k0 // spc) * nt + tile
            if item < full * G:  # full-wave item: one segment, slot (item % G, item / G)
                assert (c, idx, k0 % spc) == (item % G, item // G, 0)
            else:
                assert idx >= full
        by_finish = sorted(segs, key=lambda s: (s[0] // spc, s[2]))  # chunk, then CTA
        assert by_finish == segs
