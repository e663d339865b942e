"""Writes tests/golden/std_sort.npz: the order in which libstdc++'s std::sort leaves cubes with equal beg_t keys.

CollisionCheck sorts its cubes with std::sort(temp.begin(), temp.end(), beg_t <) (solve_3d.cc:630).  std::sort is not
stable past 16 elements, so the order of equal keys is whatever libstdc++'s introsort makes of them; the oracle restates
that algorithm (oracle_std_sort_by_beg_t).  This script compiles the real std::sort with that comparator on the oracle's
112-byte cube record, runs it on the key sets of tests/test_oracle_golden.py::test_std_sort_restatement_equals_libstdcxx
and stores keys + resulting permutations, so that the test needs no C++ toolchain and no reference build.

    python oracle/gen_std_sort_golden.py      (g++ with libstdc++)
"""
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

SRC = r"""
#include <algorithm>
#include <cstdio>
#include <vector>
#include "spectral_oracle.h"
int main() {
  int n;
  while (std::scanf("%d", &n) == 1) {
    std::vector<OracleCube> c(n);
    for (int i = 0; i < n; i++) {
      if (std::scanf("%d", &c[i].beg_t) != 1) return 1;
      c[i].count = i;
    }
    std::sort(c.begin(), c.end(), [](const OracleCube &r1, const OracleCube &r2) -> bool { return r1.beg_t < r2.beg_t; });
    for (int i = 0; i < n; i++) std::printf("%d ", c[i].count);
    std::printf("\n");
  }
  return 0;
}
"""


def key_sets():
    """The key sets of the test: sizes around the introsort threshold (16), eight distinct keys, many ties."""
    rng = np.random.default_rng(3)
    out = []
    for n in (1, 2, 5, 16, 17, 23, 40, 64):
        for _ in range(6):
            out.append(rng.integers(0, 8, n).astype(np.int32) * 10)
    return out


def main():
    keys = key_sets()
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "std_sort.cpp"), os.path.join(tmp, "std_sort")
        with open(src, "w") as f:
            f.write(SRC)
        subprocess.run(["g++", "-O2", "-std=c++17", "-I", HERE, "-o", exe, src], check=True)
        text = "".join("%d %s\n" % (len(k), " ".join(str(int(v)) for v in k)) for k in keys)
        lines = subprocess.run([exe], input=text, capture_output=True, text=True, check=True).stdout.splitlines()
    out = {}
    for c, (k, line) in enumerate(zip(keys, lines)):
        out["case%02d/keys" % c] = k
        out["case%02d/perm" % c] = np.array([int(v) for v in line.split()], dtype=np.int32)
    assert len(lines) == len(keys)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "std_sort.npz"), n_cases=len(keys), **out)


if __name__ == "__main__":
    main()
