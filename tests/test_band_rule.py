"""CPU check of the rule by which the blocked RBF kernels skip tiles of K(theta) (kernels_chol.cuh, tile_zero): every
element of every tile that the rule calls zero must evaluate to exactly 0.0 under the generator's own arithmetic,
sig2 * gpbo_exp_neg(-0.5 * (d * d)) with d = t_r / ell - t_c / ell, and so must the gradient term sig2 R d^2 of
lauum_grad_kernel.  The rule and the per-block intervals over the real rows are restated here in
C++ against the host build of fastmath.h (as in test_fastmath.py), over a sweep of ell, sorted, shuffled and
block-permuted abscissae, sizes that do not fill the last 128-row block, and blocks placed just across the threshold."""
import os
import re
import shutil
import subprocess
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = textwrap.dedent(r'''
    #include "fastmath.h"
    #include <algorithm>
    #include <cmath>
    #include <cstdio>
    #include <random>
    #include <vector>
    constexpr int TB = 128;
    // restatement of kernels_chol.cuh: tile_zero and the block intervals of prep_pairs_kernel
    static bool tile_zero(double lo_i, double hi_i, double lo_k, double hi_k) {
        return (lo_i - hi_k > BAND_GAP || lo_k - hi_i > BAND_GAP) && std::fmax(hi_i - lo_k, hi_k - lo_i) < BAND_SPAN_MAX;
    }
    long tiles = 0, skipped = 0, elems = 0, nonzero = 0;
    static void check(const std::vector<double>& t, double ell, double sig2) {
        const int m = (int)t.size(), T = (m + TB - 1) / TB;
        std::vector<double> x(m), lo(T, INFINITY), hi(T, -INFINITY);
        for (int i = 0; i < m; ++i) {
            x[i] = t[i] / ell;
            lo[i / TB] = std::fmin(lo[i / TB], x[i]);
            hi[i / TB] = std::fmax(hi[i / TB], x[i]);
        }
        for (int i = 0; i < T; ++i)
            for (int k = 0; k < T; ++k) {
                if (k == i) continue;
                ++tiles;
                if (!tile_zero(lo[i], hi[i], lo[k], hi[k])) continue;
                ++skipped;
                for (int r = i * TB; r < std::min(m, (i + 1) * TB); ++r)
                    for (int c = k * TB; c < std::min(m, (k + 1) * TB); ++c) {
                        const double d = x[r] - x[c], d2 = d * d;
                        const double kr = sig2 * gpbo::gpbo_exp_neg(-0.5 * d2);
                        ++elems;
                        if (kr != 0.0 || kr * d2 != 0.0 || std::signbit(kr)) ++nonzero;
                    }
            }
    }
    int main() {
        std::mt19937_64 rng(11);
        std::uniform_real_distribution<double> U(0.0, 1.0);
        const int sizes[] = {1000, 2048, 1500};
        for (int m : sizes) {
            std::vector<double> t(m);
            for (int i = 0; i < m; ++i) t[i] = (double)i / (m - 1);
            std::vector<double> ts = t;                  // sorted grid
            std::vector<double> tr(m);
            for (double& v : tr) v = U(rng);             // random, unsorted
            std::vector<double> tsh = t;
            std::shuffle(tsh.begin(), tsh.end(), rng);   // shuffled grid
            // unsorted but block-local: the grid's 128-point runs in shuffled order, each run shuffled as well
            const int T = (m + TB - 1) / TB;
            std::vector<int> perm(T);
            for (int b = 0; b < T; ++b) perm[b] = b;
            std::shuffle(perm.begin(), perm.end(), rng);
            std::vector<double> tb;
            for (int b : perm) {
                std::vector<double> run(t.begin() + b * TB, t.begin() + std::min(m, (b + 1) * TB));
                std::shuffle(run.begin(), run.end(), rng);
                tb.insert(tb.end(), run.begin(), run.end());
            }
            for (int q = 0; q <= 20; ++q) {
                const double ell = std::pow(10.0, -5.0 + 4.0 * q / 20.0);      // 1e-5 ... 1e-1
                check(ts, ell, 2.5);
                check(tr, ell, 0.7);
                check(tsh, ell, 1.0);
                check(tb, ell, 3.0);
            }
        }
        // blocks just across the threshold: block 0 at 0, block 1 at BAND_GAP (+- a few ulp) with ell = 1
        for (int s = -4; s <= 4; ++s) {
            std::vector<double> t(2 * TB, 0.0);
            double g = BAND_GAP;
            for (int q = 0; q < std::abs(s); ++q) g = std::nextafter(g, s > 0 ? INFINITY : 0.0);
            for (int r = TB; r < 2 * TB; ++r) t[r] = g;
            check(t, 1.0, 1.0);
        }
        std::printf("%ld %ld %ld %ld\n", tiles, skipped, elems, nonzero);
    }
''')


def band_constants():
    """The rule's constants as the device code defines them (kernels_chol.cuh)."""
    with open(os.path.join(ROOT, "gp-bayesopinf_b200", "csrc", "kernels_chol.cuh")) as f:
        src = f.read()
    return {n: re.search(rf"constexpr double {n} = ([0-9.eE+-]+);", src).group(1) for n in ("BAND_GAP", "BAND_SPAN_MAX")}


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_skipped_tiles_are_exactly_zero(tmp_path):
    src = tmp_path / "band.cpp"
    src.write_text(SRC)
    exe = tmp_path / "band"
    inc = os.path.join(ROOT, "gp-bayesopinf_b200", "csrc")
    defs = [f"-D{n}={v}" for n, v in band_constants().items()]
    subprocess.run(["g++", "-O2", "-mfma", "-ffp-contract=off", *defs, "-I", inc, "-o", str(exe), str(src)], check=True)
    tiles, skipped, elems, nonzero = map(int, subprocess.run([str(exe)], check=True, capture_output=True,
                                                                          text=True).stdout.split())
    assert nonzero == 0                  # every element of every skipped tile is +0.0, its gradient term too
    assert skipped > tiles // 4          # not vacuous: short length scales skip most tiles of block-local t
    assert elems > 10_000_000
