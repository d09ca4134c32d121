"""The matcher's kernel choice and launch sizes, from the host code frb_match itself runs (no GPU needed).

A few lines of host C++ against match_kernel.cuh print match_plan() and the dynamic shared memory of both kernels for
a grid of (l1, l2, n, rows) and for every case of the GPU matcher tests (matcher_cases.py): each of those must reach
the kernels it is named for, and every launch must fit the shared memory its kernel is allowed."""
import os
import re
import shutil
import subprocess
import tempfile

import pytest

import matcher_cases as MC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "frender_b200", "csrc")
PATHS = {0: "cand", 1: "sweep", 2: "wide"}
B200_SMEM_OPTIN = 227 * 1024      # largest dynamic shared memory a block can opt into on sm_100
STATIC_SMEM = 48 * 1024           # what a kernel gets without cudaFuncSetAttribute


def doc_rule(rows, l1, l2, n, wide):
    """The selection rule as documented: candidate tables when the context is narrow, the sheet has rows and two
    indexes, each index has at most 10 symbols and at least n + 1, n <= 3 and rows * (n + 1) * 2 <= 4096; 2048 slots
    up to rows * (n + 1) * 2 = 2048, else 4096.  Everything else narrow sweeps."""
    if wide:
        return "wide", 0
    need = rows * (n + 1) * 2
    if rows > 0 and l2 > 0 and l1 <= 10 and l2 <= 10 and n <= 3 and n + 1 <= min(l1, l2) and need <= 4096:
        return "cand", 2048 if need <= 2048 else 4096
    return "sweep", 0


@pytest.fixture(scope="module")
def plan():
    """query (rows, l1, l2, n, wide, rc) -> (path, slots, blocks_per_sm, smem of kernel 1, smem of kernel 2), and the
    header's constants."""
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    nvcc = shutil.which("nvcc") or os.path.join(cuda, "bin", "nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    queries = set()
    for _, l1, l2, n, rows, wide, _, _ in MC.plan_cases():
        queries.add((rows, l1, l2, n, wide, 1 if l2 else 0))
    lengths = [1, 2, 3, 4, 5, 6, 8, 9, 10, 11, 12, 19, 20]
    row_grid = [0, 1, 2, 48, 255, 256, 257, 341, 342, 512, 513, 682, 683, 1024, 1025, 2048, 2049, 4096, 5000]
    for l1 in lengths:
        for l2 in [0] + lengths:
            if l1 + (l2 + 1 if l2 else 0) > 21:            # the narrow sheet loader's limit
                continue
            for n in range(6):
                for rows in row_grid:
                    queries.add((rows, l1, l2, n, False, 0))
    for n in range(4):                          # the candidate kernels at every usable row count, rc pass
        for rows in range(1, 4096 // (2 * (n + 1)) + 1):
            queries.add((rows, 10, 10, n, False, 1))
    for wide in (False, True):
        queries.add((MC.MAX_ROWS, 10, 10, 1, wide, 1))
    queries = sorted(queries)
    body = ",\n".join(f"{{{r}u, {a}u, {b}u, {n}u, {int(w)}, {rc}}}" for r, a, b, n, w, rc in queries)
    src = ('#include <cstdio>\n#include "match_kernel.cuh"\n'
           "struct Q { unsigned rows, l1, l2, n; int wide, rc; };\n"
           f"static const Q qs[] = {{\n{body}\n}};\n"
           "int main() {\n"
           '    std::printf("%d %d %d\\n", frb::kMatchSmemMax, frb::kMatchWideSmemMax, frb::kMatchThreads);\n'
           "    for (const Q& q : qs) {\n"
           "        const frb::MatchPlan p = frb::match_plan(q.rows, q.l1, q.l2, q.n, q.wide != 0);\n"
           '        std::printf("%d %u %d %zu %zu\\n", static_cast<int>(p.path), p.slots, p.blocks_per_sm,\n'
           "                    frb::match_smem_idx1(p, q.rows, q.n), frb::match_smem_classify(p, q.rows, q.n, q.rc != 0));\n"
           "    }\n    return 0;\n}\n")
    tmp = tempfile.mkdtemp(prefix="frb_match_plan_")
    try:
        with open(os.path.join(tmp, "plan.cu"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "plan")
        subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", f"-I{CSRC}", "-x", "cu",
                        os.path.join(tmp, "plan.cu"), "-o", exe], check=True, capture_output=True)
        lines = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    limit, wide_limit, threads = map(int, lines[0].split())
    out = {}
    for q, line in zip(queries, lines[1:]):
        path, slots, bps, s1, s2 = map(int, line.split())
        out[q] = (PATHS[path], slots, bps, s1, s2)
    assert len(out) == len(queries)
    return out, {"limit": limit, "wide_limit": wide_limit, "threads": threads}


def test_gpu_cases_take_the_kernels_they_are_named_for(plan):
    got, _ = plan
    for label, l1, l2, n, rows, wide, path, slots in MC.plan_cases():
        p = got[(rows, l1, l2, n, wide, 1 if l2 else 0)]
        assert p[0] == path, (label, p)
        if slots is not None:
            assert p[1] == slots, (label, p)
    # every boundary case sits right next to a change of path or table size
    for n, rows, path, slots in MC.BOUNDARY:
        if rows not in (1, MC.MAX_ROWS):
            around = {doc_rule(rows - 1, 10, 10, n, False), doc_rule(rows + 1, 10, 10, n, False)}
            assert around != {(path, slots)}, (n, rows)


def test_selection_rule(plan):
    """match_plan over lengths 1..20 (single and dual index), n = 0..5 and row counts around every threshold
    against the documented rule."""
    got, _ = plan
    for (rows, l1, l2, n, wide, rc), p in got.items():
        assert (p[0], p[1]) == doc_rule(rows, l1, l2, n, wide), ((rows, l1, l2, n, wide), p)


def test_launches_fit_their_shared_memory(plan):
    """Every launch fits the shared memory its kernel is allowed: the candidate kernels at every usable shape (rc
    pass, two tables), match_kernel and match_wide_kernel at 5000 rows, and kernel 1 of the sweep / wide paths, which
    has no attribute, in the default 48 KiB; the grids stay within the sm_count x 8 blocks the GPU tests size their
    scale cases by."""
    got, k = plan
    assert k["threads"] == MC.GRID_THREADS_PER_BLOCK
    assert k["limit"] == 200 * 1024 and k["wide_limit"] == 220 * 1024
    assert k["limit"] <= B200_SMEM_OPTIN and k["wide_limit"] <= B200_SMEM_OPTIN
    seen = {"cand": 0, "sweep": 0, "wide": 0}
    for (rows, l1, l2, n, wide, rc), (path, slots, bps, s1, s2) in got.items():
        assert 1 <= bps <= MC.GRID_BLOCKS_PER_SM
        if path == "cand":
            assert s1 <= k["limit"] and s2 <= k["limit"], (rows, n, s1, s2)
        else:
            assert s1 <= STATIC_SMEM, (path, rows, s1)
            assert s2 <= (k["wide_limit"] if path == "wide" else k["limit"]), (path, rows, s2)
        seen[path] = max(seen[path], s2)
    assert got[(MC.MAX_ROWS, 10, 10, 1, False, 1)][4] == 180_016      # 5000 x (4 x 8 + 4) + 16
    assert got[(MC.MAX_ROWS, 10, 10, 1, True, 1)][4] == 220_016       # 5000 x (5 x 8 + 4) + 16
    assert seen["cand"] > 100 * 1024                                   # the largest tables were among the queries


def test_frb_match_launches_from_the_plan():
    """frb_match takes its kernels, grids and shared memory from match_plan, and the attributes from the header."""
    src = open(os.path.join(CSRC, "frb_lib.cu")).read()
    body = src[src.index("int frb_match("):src.index("int frb_demux_ok(")]
    assert "match_plan(c->rows, c->l1, c->l2, n_subs, c->wide)" in body
    assert len(re.findall(r"<<<grid, kMatchThreads, smem[12], c->compute>>>", body)) == 6
    for kern, lim in (("match_kernel", "kMatchSmemMax"), ("match_cand_kernel", "kMatchSmemMax"),
                      ("match_idx1_cand_kernel", "kMatchSmemMax"), ("match_wide_kernel", "kMatchWideSmemMax")):
        assert f"cudaFuncSetAttribute({kern}, cudaFuncAttributeMaxDynamicSharedMemorySize, {lim})" in src
