// persist_geometry.h -- shared-memory geometry of the device-resident solve (persist.cuh): the block length of the tiled S/Y
// history and the number of stages each staged pass fits into the kernel's staging ring.  The kernel sizes its passes with these
// functions and the host (persist_host.cuh) picks the block length and refuses a configuration in which some pass would get no
// stage at all (it would wait for a bulk copy that was never issued).  Plain C++: the header also compiles without CUDA, so that
// the whole table can be checked on a CPU (tests/test_persist_geometry_cpu.py).
#pragma once

#if defined(__CUDACC__)
#define LB_GEOM_HD __host__ __device__
#else
#define LB_GEOM_HD
#endif

namespace lb {

constexpr int kPStageBytes = 196608;   // dynamic shared memory of the persistent kernel: the staging ring of its staged passes
constexpr int kPMaxStages = 4;         // stages (mbarriers) a staged pass may use
constexpr int kTrialTE = 2016;         // tile of the neighbour-coupled trial pass: 63 x 32 elements
constexpr int kPBlockMax = 1024, kPBlockMin = 32;

// Block length BT of the tiled history: the largest power of two in [32, 1024] for which `want_stages` stages of 2m+4 rows of BT
// elements fit the staging ring (2m+4: the fused combination pass of the tridiagonal quadratic, g, x, two data vectors, 2m columns).
LB_GEOM_HD constexpr int persist_block_len(int m, int elem_bytes, int want_stages)
{
    int bt = kPBlockMax;
    while (bt > kPBlockMin && (long long)want_stages * (2 * m + 4) * bt * elem_bytes > kPStageBytes) bt >>= 1;
    return bt;
}

// stages of a pass that stages `stage_elems` elements per tile (0: not even one tile fits)
LB_GEOM_HD constexpr int persist_stages(long long stage_elems, int elem_bytes)
{
    const long long s = (long long)kPStageBytes / (stage_elems * elem_bytes);
    return s > kPMaxStages ? kPMaxStages : (int)s;
}

// p_dots: the right-hand vectors (FORM: g, x, gp, xp; PLAIN: g) and 2 rows per old history column
LB_GEOM_HD constexpr int dots_stages(int elem_bytes, int bt, bool form, int cnt_old)
{
    return persist_stages((long long)((form ? 4 : 1) + 2 * cnt_old) * bt, elem_bytes);
}

// p_combine: g (, x for the fused first trial) (, the objective's data vectors when it is neighbour-coupled), 2 rows per column, and
// for a neighbour-coupled objective one 16-byte granule on either side of the x row
LB_GEOM_HD constexpr int combine_stages(int elem_bytes, int bt, int c, bool fuse, bool halo, int data_vectors)
{
    const int rows = (fuse ? 2 : 1) + (halo ? data_vectors : 0) + 2 * c;
    return persist_stages((long long)rows * bt + (halo ? 2 * (16 / elem_bytes) : 0), elem_bytes);
}

// p_trial_halo: `nin` input vectors (FIRST: x; TRIAL: xp, d) and the data vectors, each a kTrialTE tile with a granule on either side
LB_GEOM_HD constexpr int trial_halo_stages(int elem_bytes, int nin, int data_vectors)
{
    return persist_stages((long long)(nin + data_vectors) * (kTrialTE + 2 * (16 / elem_bytes)), elem_bytes);
}

// The fewest stages any pass of a solve gets (history size m, block length bt, objective coupled to its neighbours or not, with
// `data_vectors` data vectors).  Stage counts only fall as the number of columns c grows, so the full ring (c = m) decides:
// the pair-forming dots pass sees at most m - 1 old columns, the plain one and the combination pass m.
LB_GEOM_HD constexpr int persist_min_stages(int m, int elem_bytes, int bt, bool halo, int data_vectors)
{
    int s = dots_stages(elem_bytes, bt, true, m - 1);
    const int cand[3] = {dots_stages(elem_bytes, bt, false, m), combine_stages(elem_bytes, bt, m, true, halo, data_vectors),
                         combine_stages(elem_bytes, bt, m, false, false, 0)};
    for (int k = 0; k < 3; k++) s = cand[k] < s ? cand[k] : s;
    if (halo)
    {
        const int t0 = trial_halo_stages(elem_bytes, 1, data_vectors), t1 = trial_halo_stages(elem_bytes, 2, data_vectors);
        s = t0 < s ? t0 : s;
        s = t1 < s ? t1 : s;
    }
    return s;
}

}  // namespace lb
