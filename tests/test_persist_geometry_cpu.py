"""The shared-memory geometry of the device-resident solve (lbfgspp_b200/csrc/persist_geometry.h), compiled with g++ and checked on
the CPU: every configuration the host accepts gives every staged pass at least one stage (a pass without one would wait for a bulk
copy that was never issued), the default history block lengths are the ones the solver has always used, and the Python mirror that
test_gpu_persist_edges.py builds its cases from agrees with the header."""
import os
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "lbfgspp_b200", "csrc", "persist_geometry.h")

# the host's choice (persist_host.cuh, lbfgs_b200_solver_create_batch): want_stages = 2 unless LBFGS_B200_STAGES is 1..4;
# objectives 0..3 = paired Rosenbrock, shifted quadratic, chained Rosenbrock, tridiagonal quadratic
PROGRAM = r"""
#include <cstdio>
#include "persist_geometry.h"
using namespace lb;
int main()
{
    for (int elem = 4; elem <= 8; elem += 4)
        for (int env = 0; env <= 4; env++)
            for (int m = 1; m <= 64; m++)
                for (int obj = 0; obj < 4; obj++)
                {
                    const int want = env == 0 ? 2 : env;
                    const int bt = persist_block_len(m, elem, want);
                    const bool halo = obj >= 2;
                    const int dv = obj == 3 ? 2 : 0;
                    int dmin = 99, cmin = 99;
                    for (int c = 0; c <= m; c++)   // every ring fill the solve goes through
                    {
                        const int a = c >= 1 ? dots_stages(elem, bt, true, c - 1) : 99, b = dots_stages(elem, bt, false, c);
                        const int f = combine_stages(elem, bt, c, true, halo, dv), u = combine_stages(elem, bt, c, false, false, 0);
                        dmin = a < dmin ? a : dmin; dmin = b < dmin ? b : dmin;
                        cmin = f < cmin ? f : cmin; cmin = u < cmin ? u : cmin;
                    }
                    const int t = halo ? (trial_halo_stages(elem, 1, dv) < trial_halo_stages(elem, 2, dv) ? trial_halo_stages(elem, 1, dv)
                                                                                                         : trial_halo_stages(elem, 2, dv)) : 99;
                    const int fused_full = combine_stages(elem, bt, m, true, halo, dv);
                    std::printf("%d %d %d %d %d %d %d %d %d %d\n", elem, env, m, obj, bt, dmin, cmin, t, fused_full,
                                persist_min_stages(m, elem, bt, halo, dv));
                }
    return 0;
}
"""


@pytest.fixture(scope="module")
def table():
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "geom.cpp"), os.path.join(tmp, "geom")
        with open(src, "w") as f:
            f.write(PROGRAM)
        subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), "-o", exe, src], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    rows = {}
    for line in out.split("\n"):
        if line:
            elem, env, m, obj, bt, dmin, cmin, t, fused_full, least = map(int, line.split())
            rows[(elem, env, m, obj)] = dict(bt=bt, dots=dmin, combine=cmin, trial=t, fused_full=fused_full, least=least)
    assert len(rows) == 2 * 5 * 64 * 4
    return rows


def test_accepted_configurations_stage_every_pass(table):
    for key, r in table.items():
        # the host refuses the solve when persist_min_stages < 1; whatever it accepts must stage every pass at every ring fill
        assert r["least"] == min(r["dots"], r["combine"], r["trial"]), key
        if r["least"] >= 1:
            assert min(r["dots"], r["combine"], r["trial"]) >= 1, key


def test_default_block_length_stages_everything(table):
    for (elem, env, m, obj), r in table.items():
        if env == 0:
            assert r["least"] >= 1, (elem, m, obj)


def test_single_stage_knob_is_refused_exactly_where_the_margin_does_not_fit(table):
    """LBFGS_B200_STAGES=1 sizes the blocks so that ONE stage of 2m+4 rows fills the ring; where that is exact, the two granules of
    margin of the tridiagonal quadratic's fused pass no longer fit and the host must refuse the solve (no GPU run needed)."""
    refused = sorted((elem, m, obj) for (elem, env, m, obj), r in table.items() if r["least"] < 1)
    assert all(table[(elem, 1, m, obj)]["least"] == 0 for elem, m, obj in refused)
    assert {(elem, env) for (elem, env, m, obj), r in table.items() if r["least"] < 1} <= {(4, 1), (8, 1)}
    assert refused == sorted([(8, m, 3) for m in (10, 22, 46)] + [(4, m, 3) for m in (22, 46)])


def test_default_block_length_table_is_pinned(table):
    """The block lengths the solver uses by default (a change here moves every resident result's summation order)."""
    pinned = {8: [(range(1, 5), 1024), (range(5, 11), 512), (range(11, 23), 256), (range(23, 47), 128), (range(47, 65), 64)],
              4: [(range(1, 11), 1024), (range(11, 23), 512), (range(23, 47), 256), (range(47, 65), 128)]}
    for elem, spans in pinned.items():
        for ms, bt in spans:
            for m in ms:
                for obj in range(4):
                    assert table[(elem, 0, m, obj)]["bt"] == bt, (elem, m)


def test_single_stage_pass_is_reached_by_default(table):
    """The configurations whose full-ring fused combination pass runs on ONE stage with the default blocks (tridiagonal quadratic:
    fp64 m in {4, 10, 22, 46}, fp32 m in {10, 22, 46})."""
    one = sorted((elem, m) for (elem, env, m, obj), r in table.items() if env == 0 and obj == 3 and r["fused_full"] == 1)
    assert one == sorted([(8, m) for m in (4, 10, 22, 46)] + [(4, m) for m in (10, 22, 46)])


def test_python_mirror_agrees_with_header(table):
    import test_gpu_persist_edges as edges
    for (elem, env, m, obj), r in table.items():
        if env == 0:
            assert edges.block_len(m, elem) == r["bt"], (elem, m)
            st = edges.stage_counts(m, elem, obj)
            assert st["least"] == r["least"] and st["fused_full"] == r["fused_full"], (elem, m, obj, st, r)
