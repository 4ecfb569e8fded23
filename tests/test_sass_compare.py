"""tools/sass_compare.py maps the demangled names of every kernel naming scheme to one key (no build needed)."""
import importlib.util
import os

import pytest

_PATH = os.path.join(os.path.dirname(__file__), "..", "tools", "sass_compare.py")
_spec = importlib.util.spec_from_file_location("sass_compare", _PATH)
sass_compare = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sass_compare)


@pytest.mark.parametrize(
    "name, key",
    [
        # before weights: no mode argument
        ("void vsr::fit_kernel<double, 3, 2>(vsr::FitArgs)", ("fit_kernel", "double", 3, 2, "linear")),
        ("void vsr::gram_kernel<16, 1>(vsr::GramArgs)", ("gram_kernel", "double", 16, 1, "linear")),
        # <..., W>
        ("void vsr::eval_kernel<float, 4, 2, true>(vsr::Weighted<vsr::EvalArgs, true>)",
         ("eval_kernel", "float", 4, 2, "weighted")),
        ("void vsr::gram_kernel<2, 2, false>(vsr::Weighted<vsr::GramArgs, false>)",
         ("gram_kernel", "double", 2, 2, "linear")),
        # <..., W, RB>
        ("void vsr::eval_tile_kernel<double, 12, 1, false, false>(std::conditional<false, "
         "vsr::Robust<vsr::EvalTileArgs>, vsr::Weighted<vsr::EvalTileArgs, false> >::type)",
         ("eval_tile_kernel", "double", 12, 1, "linear")),
        ("void vsr::gram_kernel<1, 2, true, false>(std::conditional<false, vsr::Robust<vsr::GramArgs>, "
         "vsr::Weighted<vsr::GramArgs, true> >::type)", ("gram_kernel", "double", 1, 2, "weighted")),
        ("void vsr::fit_kernel<float, 0, 2, false, true>(std::conditional<true, vsr::Robust<vsr::FitArgs>, "
         "vsr::Weighted<vsr::FitArgs, false> >::type)", ("fit_kernel", "float", 0, 2, "robust")),
        # (vsr::LossMode)n
        ("void vsr::eval_kernel<double, 1, 2, (vsr::LossMode)0>(vsr::LaunchArgs<vsr::EvalArgs, (vsr::LossMode)0>)",
         ("eval_kernel", "double", 1, 2, "linear")),
        ("void vsr::gram_kernel<8, 2, (vsr::LossMode)1>(vsr::LaunchArgs<vsr::GramArgs, (vsr::LossMode)1>)",
         ("gram_kernel", "double", 8, 2, "weighted")),
        ("void vsr::fit_kernel<float, 3, 2, (vsr::LossMode)2>(vsr::LaunchArgs<vsr::FitArgs, (vsr::LossMode)2>)",
         ("fit_kernel", "float", 3, 2, "robust")),
        # predict_kernel has no mode in any scheme
        ("void vsr::predict_kernel<float, 16, 1>(vsr::PredictArgs)", ("predict_kernel", "float", 16, 1, "linear")),
    ],
)
def test_kernel_key(name, key):
    assert sass_compare.kernel_key(name) == key


@pytest.mark.parametrize(
    "name",
    [
        "void vsr::eval_finalize(double const*, int const*, int const*, int const*, int, int, int, int, double, "
        "double*, double*)",
        "void vsr::fill_nan_rows(int const*, int, int, double*)",
    ],
)
def test_other_functions_are_skipped(name):
    assert sass_compare.kernel_key(name) is None


def test_unknown_scheme_is_an_error():
    with pytest.raises(ValueError):
        sass_compare.kernel_key("void vsr::fit_kernel<double, 1, 2, 7, 8, 9>(vsr::FitArgs)")
