"""The kernel set a context runs (csrc/tables.cpp plan_run), on the CPU through the tables shim: every configuration whose
kernel set a GPU test asserts names the same set here, read from those tests' own case tables, and the edges of each rule."""
import ctypes as C

import pytest

import test_gpu_narrow
import test_gpu_native
import test_gpu_pipeline
import test_gpu_tile_aux
import test_gpu_tile_m2
from test_tables import shim  # noqa: F401  (the fixture that builds tests/tables_shim.cpp)
from vcfgl_b200 import args as vargs
from vcfgl_b200 import capi

SAMPLER_PER_READ, SAMPLER_COUNTS = 1, 2      # include/vgl.h VGL_SAMPLER_*
PER_READ = "k_sim+k_site+k_scan+k_emit"
FUSED, TILE, TILE_M2, TRUTH = "k_fused_m1f", "k_tile_m1f", "k_tile_m2", "k_truth_site+k_scan+k_truth_emit"
STATS = test_gpu_native.STATS
DF_DEPTHS = [0.5 + (i % 5) * 2.0 for i in range(37)]      # test_gpu_tile_m2.test_tile_kernels_with_per_sample_depths


@pytest.fixture(scope="module")
def plan(shim):  # noqa: F811
    f = shim.shim_kernel_set
    f.argtypes = [C.POINTER(capi.VglParams), C.c_int, C.POINTER(C.c_int)]
    f.restype = C.c_char_p

    def call(argv, S, B, sampler=0, allow_tile=True, qs_bins=None, depths=None, fixed_depth=False, status=capi.VGL_OK):
        a = vargs.parse_args(argv if isinstance(argv, list) else argv.split(), qs_bins=qs_bins, depths=depths)
        p = capi.params_from_args(a, S, max_batch_sites=B, n_slots=1, sampler=sampler, fixed_depth=fixed_depth)
        rc = C.c_int(1)
        name = f(C.byref(p), int(allow_tile), C.byref(rc)).decode()
        assert rc.value == status
        return name
    return call


def stats_case(name, drop_strand=False):
    """test_gpu_native.distributions(): the fixture's command line, S and batch size"""
    st = STATS[name]
    argv = list(st["argv"])
    if drop_strand:
        for flag in ("-addFormatADF", "-addFormatADR"):
            while flag in argv:
                i = argv.index(flag)
                del argv[i:i + 2]
    return argv, st["S"], min(2000 * 100 // st["S"], st["n_sites"]), dict(qs_bins=st.get("qs_bins"), depths=st.get("depths"))


@pytest.mark.parametrize("name,sampler,kernels,drop_strand", test_gpu_native.DIST_RUNS)
def test_native_distribution_runs(plan, name, sampler, kernels, drop_strand):
    argv, S, B, kw = stats_case(name, drop_strand)
    assert plan(argv, S, B, sampler=sampler, **kw) == kernels


def test_native_fixed_depth(plan):
    argv, S, B, kw = stats_case("gl1_d10", drop_strand=True)
    assert plan(argv, S, B, fixed_depth=True, **kw) == TILE


@pytest.mark.parametrize("name,allow_tile,kernels", [("gl1_d10", False, FUSED), ("gl1_d10", True, TILE), ("gl1_d30", False, FUSED),
                                                     ("gl1_d30", True, TILE), ("gl1_df", False, FUSED), ("gl1_df", True, TILE)])
def test_fused_count_sampler_runs(plan, name, allow_tile, kernels):
    """test_gpu_fused.test_count_sampler_distributions_match_reference (VGL_NO_TILE: allow_tile = False)"""
    st = STATS[name]
    assert plan(st["argv"], st["S"], 2000, sampler=SAMPLER_COUNTS, allow_tile=allow_tile, depths=st.get("depths")) == kernels


@pytest.mark.parametrize("name", sorted(test_gpu_tile_m2.CASES))
def test_tile_m2_cases(plan, name):
    argv, S, n_sites, bins = test_gpu_tile_m2.CASES[name]
    assert plan(argv, S, n_sites, qs_bins=bins) == TILE_M2


@pytest.mark.parametrize("argv,kernels", [("--seed 31 -e 0.05 -GL 2 -addPL 1 -addFormatAD 1", TILE_M2),
                                          ("--seed 32 -e 0.01 -eq 2 -bv 1e-4 -GL 2 -addPL 1 -addFormatAD 1", TILE_M2),
                                          ("--seed 33 -e 0.02 -GL 1 -addPL 1 -addFormatAD 1", TILE),
                                          ("--seed 34 -e 0.02 -GL 1 -addPL 1 -addI16 1 -addQS 1", TILE)])
@pytest.mark.parametrize("B", [400, 4000])
def test_tile_kernels_with_per_sample_depths(plan, argv, kernels, B):
    assert plan(argv, 37, B, depths=DF_DEPTHS) == kernels


@pytest.mark.parametrize("name", sorted(test_gpu_tile_aux.CASES))
def test_tile_aux_cases(plan, name):
    argv, S, n_sites = test_gpu_tile_aux.CASES[name]
    assert plan(argv, S, n_sites) == TILE


def test_tile_aux_strand_laws(plan):
    assert plan("--seed 21 -d 10 -e 0.01 -GL 1 -doUnobserved 1 -addPL 1 -addI16 1 -addInfoAD 1 -addInfoADF 1 -addInfoADR 1", 50, 4000) == TILE


@pytest.mark.parametrize("u", range(6))
def test_truth(plan, u):
    assert plan("--seed 1 --depth inf -e 0 -GL 1 -doUnobserved %d -addGL 1 -addGP 1 -addPL 1 -addFormatDP 0" % u, 37, 150) == TRUTH


@pytest.mark.parametrize("name", sorted(test_gpu_pipeline.CASES))
def test_pipeline_cases(plan, name):
    argv, S, B, kernels, bins = test_gpu_pipeline.CASES[name]
    assert plan(argv, S, B, qs_bins=bins) == kernels


@pytest.mark.parametrize("name", sorted(k for k, v in test_gpu_narrow.NATIVE.items() if v[3]))
def test_narrow_cases(plan, name):
    argv, S, n_sites, kernels, _ = test_gpu_narrow.NATIVE[name]
    assert plan(argv, S, n_sites) == kernels


# ---- the edges of the rules
GL1 = "--seed 3 -d 10 -e 0.01 -GL 1 -addPL 1 -addFormatAD 1"
GL2 = "--seed 4 -d 6 -e 0.01 -GL 2 -addPL 1 -addFormatAD 1"


@pytest.mark.parametrize("argv,tile", [(GL1, TILE), (GL2, TILE_M2)])
def test_tile_sample_limit(plan, argv, tile):
    assert plan(argv, 60000, 1) == tile
    assert plan(argv, 60001, 1) == (FUSED if tile == TILE else PER_READ)


@pytest.mark.parametrize("argv,tile", [(GL1, TILE), (GL2, TILE_M2)])
def test_fixed_depth_limit(plan, argv, tile):
    """a fixed depth of 256 or more does not fit the alias table's 256 columns"""
    argv = argv.replace("-d 10", "-d 6")
    assert plan(argv.replace("-d 6", "-d 255"), 4, 10, fixed_depth=True) == tile
    assert plan(argv.replace("-d 6", "-d 256"), 4, 10, fixed_depth=True) == (FUSED if tile == TILE else PER_READ)


@pytest.mark.parametrize("argv,tile", [(GL1, TILE), (GL2, TILE_M2)])
def test_poisson_mean_beyond_the_alias_table(plan, argv, tile):
    argv = argv.replace("-d 10", "-d 6")
    assert plan(argv.replace("-d 6", "-d 100"), 4, 10) == tile
    assert plan(argv.replace("-d 6", "-d 200"), 4, 10) == (FUSED if tile == TILE else PER_READ)


@pytest.mark.parametrize("argv,tile", [(GL1, TILE), (GL2, TILE_M2)])
def test_depths_file_with_a_mean_beyond_the_alias_table(plan, argv, tile):
    assert plan(argv, 37, 400, depths=DF_DEPTHS) == tile
    assert plan(argv, 37, 400, depths=DF_DEPTHS[:-1] + [200.0]) == (FUSED if tile == TILE else PER_READ)


def test_error_qs_1_under_gl1_takes_the_fused_kernel(plan):
    assert plan("--seed 9 -d 5 -e 0.05 -eq 1 -bv 1e-3 -GL 1 -addPL 1 -addFormatAD 1", 37, 150) == FUSED


def test_precise_gl_without_errors_takes_the_general_kernels(plan):
    """homT = log10(1 - 0) = 0: the model-2 tile kernel's table-driven update needs negative constants"""
    assert plan("--seed 18 -d 5 -e 0.02 -GL 2 --precise-gl 1 -addPL 1", 33, 200) == TILE_M2
    assert plan("--seed 18 -d 5 -e 0 -GL 2 --precise-gl 1 -addPL 1", 33, 200) == PER_READ


@pytest.mark.parametrize("argv", [GL1, GL2])
def test_per_read_sampler(plan, argv):
    assert plan(argv, 37, 150, sampler=SAMPLER_PER_READ) == PER_READ


def test_count_sampler_refuses_planes_of_2_31_elements(plan):
    """the G-shaped plane holds B x (15 S rounded up to 4) elements: 143165 x 15000 < 2^31 <= 143166 x 15000"""
    assert plan(GL1, 1000, 143165, sampler=SAMPLER_COUNTS) == TILE
    assert plan(GL1, 1000, 143165, sampler=SAMPLER_COUNTS, allow_tile=False) == FUSED
    plan(GL1, 1000, 143166, sampler=SAMPLER_COUNTS, status=capi.VGL_EINVAL)
    assert plan(GL1, 1000, 143166) == PER_READ
