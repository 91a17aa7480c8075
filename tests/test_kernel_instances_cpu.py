"""CPU checks of the kernel instance table (tests/kernel_instances.py): the name key on both printed forms, and that the
cases plus the exempt list cover exactly the kernel instances of the built libspx.so."""
import os

import pytest

from tests import kernel_instances as ki

# one instance of every family, as cu++filt prints it (from cuobjdump -sass) and as the CUDA profiler prints it
NAME_FORMS = [
    ("spx::stft_kernel<(int)1024, (int)0, (bool)1, (int)0, (int)2, (bool)1, (int)1>(spx::StftParams)",
     "void spx::stft_kernel<1024, 0, true, 0, 2, true, 1>(spx::StftParams)", "stft_kernel<1024, 0, true, 0, 2, true, 1>"),
    ("spx::stft2_kernel<(int)1024, (int)0, (bool)1, (int)2, (int)23>(spx::StftParams, CUtensorMap_st)",
     "void spx::stft2_kernel<1024, 0, true, 2, 23>(spx::StftParams, CUtensorMap_st)", "stft2_kernel<1024, 0, true, 2, 23>"),
    ("spx::stft2_strip_kernel<(int)0, (bool)0, (int)4, (int)2, (int)7>(spx::StftParams, CUtensorMap_st)",
     "void spx::stft2_strip_kernel<0, false, 4, 2, 7>(spx::StftParams, CUtensorMap_st)",
     "stft2_strip_kernel<0, false, 4, 2, 7>"),
    ("spx::big_cols_kernel<(int)512, (int)1024, (int)1, (bool)0>(spx::BigParams)",
     "void spx::big_cols_kernel<512, 1024, 1, false>(spx::BigParams)", "big_cols_kernel<512, 1024, 1, false>"),
    ("spx::big_rows_kernel<(int)512, (int)1024, (bool)1, (bool)1>(spx::BigParams)",
     "void spx::big_rows_kernel<512, 1024, true, true>(spx::BigParams)", "big_rows_kernel<512, 1024, true, true>"),
    ("spx::big2_kernel<(bool)1, (int)1>(spx::Big2Params, CUtensorMap_st, CUtensorMap_st)",
     "void spx::big2_kernel<true, 1>(spx::Big2Params, CUtensorMap_st, CUtensorMap_st)", "big2_kernel<true, 1>"),
    ("spx::blu_pre_kernel<(int)1>(spx::BluParams)", "void spx::blu_pre_kernel<1>(spx::BluParams)", "blu_pre_kernel<1>"),
    ("spx::blu_mul_kernel(spx::BluParams)", "spx::blu_mul_kernel(spx::BluParams)", "blu_mul_kernel"),
    ("spx::features_kernel<float>(const float *, int, int, long long, spx_feature_opts, spx_features *, int *, int)",
     "void spx::features_kernel<float>(float const*, int, int, long long, spx_feature_opts, spx_features*, int*, int)",
     "features_kernel<float>"),
    ("spx::hist2d_smem_kernel<(int)0>(const void *, long long, double, spx::HistGrid, unsigned int *, bool, int, "
     "unsigned int *, int, spx::HistConst)",
     "void spx::hist2d_smem_kernel<0>(void const*, long long, double, spx::HistGrid, unsigned int*, bool, int, "
     "unsigned int*, int, spx::HistConst)", "hist2d_smem_kernel<0>"),
    ("spx::frame_stats_kernel<(int)1>(const void *, long long, int, int, float, float *, float *)",
     "void spx::frame_stats_kernel<1>(void const*, long long, int, int, float, float*, float*)", "frame_stats_kernel<1>"),
    ("spx::stream_frame_f64_kernel<(bool)0>(const void *, int, int, const double2 *, double, double *, unsigned char *, "
     "double, double)", "void spx::stream_frame_f64_kernel<false>(void const*, int, int, double2 const*, double, double*, "
     "unsigned char*, double, double)", "stream_frame_f64_kernel<false>"),
    ("spx::pool_kernel<(bool)1>(const float *, long long, long long, int, int, long long, long long, int, double *)",
     "void spx::pool_kernel<true>(float const*, long long, long long, int, int, long long, long long, int, double*)",
     "pool_kernel<true>"),
    ("spx::ddc_jobs_kernel<(int)0>(spx::DdcParams)", "void spx::ddc_jobs_kernel<0>(spx::DdcParams)", "ddc_jobs_kernel<0>"),
    ("spx::chan_kernel<(int)1, (int)4096>(spx::ChanParams)", "void spx::chan_kernel<1, 4096>(spx::ChanParams)",
     "chan_kernel<1, 4096>"),
    ("spx::det_scan_kernel(int *, int, int *)", "spx::det_scan_kernel(int*, int, int*)", "det_scan_kernel"),
    ("spx::welch_finalize_kernel(const double *, int, double, double *, double *)",
     "spx::welch_finalize_kernel(double const*, int, double, double*, double*)", "welch_finalize_kernel"),
]


@pytest.mark.parametrize("filt,prof,want", NAME_FORMS, ids=[w for _, _, w in NAME_FORMS])
def test_key_accepts_both_name_forms(filt, prof, want):
    assert ki.key(filt) == want
    assert ki.key(prof) == want


def test_case_ids_are_unique_and_cases_are_declarative():
    ids = [c["id"] for c in ki.CASES]
    assert len(ids) == len(set(ids))
    for c in ki.CASES:
        assert c["expects"] and not (c["expects"] & ki.EXEMPT), c["id"]
        assert {ki.key(k) for k in c["expects"]} == set(c["expects"]), c["id"]     # keys are written in canonical form


@pytest.fixture(scope="module")
def built_lib():
    from sdr_iq_visualizer_b200 import _native
    path = _native.LIB_PATH
    if not os.path.exists(path):
        _native.build()
    return path


def test_every_built_instance_has_a_case(built_lib):
    """The union of every case's expected instances and the exempt measurement kernels is exactly the set of kernel
    instances in the library: a new template instance without a case, or a case naming an instance the library no longer
    builds, fails here."""
    built = {ki.key(n) for n in ki.inventory(built_lib)}
    covered = ki.covered()
    missing, surplus = sorted(built - covered), sorted(covered - built)
    print(f"{len(built)} instances built; {len(covered) - len(ki.EXEMPT)} covered by {len(ki.CASES)} cases + "
          f"{len(ki.EXEMPT)} exempt")
    print("built without a case:", missing)
    print("in a case but not built:", surplus)
    assert not missing and not surplus, f"built without a case: {missing}; in a case but not built: {surplus}"
