"""Mixed batches without a GPU: formgpu_batch_create_mixed checks every entry before any CUDA call
and names the sequence of a bad one; the host-side mixed constructors reject bad lists; the sweep
driver's variant parsing and its mapping of FORM.default_params() names onto formhost_est_params."""
import ctypes as C
import os
import sys

import pytest

from form_b200 import _capi, sweep

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "python"))


def _params_array(entries):
    return (_capi.Params * len(entries))(*entries)


def test_new_symbols_are_declared_bound_and_exported():
    for name in ("formgpu_batch_create_mixed",):
        assert name in _capi.FORMGPU_SYMBOLS
        assert hasattr(_capi.gpu_lib(), name)
    for name in ("formhost_pool_create_mixed", "formhost_batch_replay_create_mixed"):
        assert name in _capi.FORMHOST_SYMBOLS
        assert hasattr(_capi.host_lib(), name)
    assert _capi.gpu_lib().formgpu_abi_version() == 1


def test_batch_create_mixed_rejects_null_and_empty_arguments():
    lib = _capi.gpu_lib()
    h = C.c_void_p()
    arr = _params_array([_capi.default_params(16, 1800)] * 2)
    assert lib.formgpu_batch_create_mixed(None, 0, None, 2, C.byref(h)) == _capi.ERR_INVALID_ARG
    assert lib.formgpu_batch_create_mixed(arr, 0, None, 0, C.byref(h)) == _capi.ERR_INVALID_ARG
    assert lib.formgpu_batch_create_mixed(arr, 0, None, 2, None) == _capi.ERR_INVALID_ARG
    assert not h.value


@pytest.mark.parametrize("bad", [dict(neighbor_points=0), dict(num_columns=5000), dict(max_window_scans=1),
                                 dict(sigma=0.0), dict(planar_feats_per_sector=-1)])
def test_batch_create_mixed_names_the_bad_sequence_before_touching_the_gpu(bad):
    lib = _capi.gpu_lib()
    h = C.c_void_p()
    entries = [_capi.default_params(16, 1800), _capi.default_params(64, 1024),
               _capi.default_params(128, 1024, **bad), _capi.default_params(64, 1024)]
    rc = lib.formgpu_batch_create_mixed(_params_array(entries), 0, None, len(entries), C.byref(h))
    assert rc in (_capi.ERR_UNSUPPORTED, _capi.ERR_INVALID_ARG), bad
    assert not h.value
    msg = lib.formgpu_batch_last_error(None)
    assert b"sequence 2" in msg, msg
    # the same entry fails the same way through formgpu_create
    assert lib.formgpu_create(C.byref(entries[2]), 0, None, C.byref(h)) == rc


def test_host_mixed_constructors_reject_bad_lists():
    lib = _capi.host_lib()
    a = _capi.default_est_params(16, 1800)
    b = _capi.default_est_params(64, 1024, device=1)
    arr = (_capi.EstParams * 2)(a, b)
    assert not lib.formhost_pool_create_mixed(arr, 2, 200)
    assert b"device" in lib.formhost_last_error() and b"sequence 1" in lib.formhost_last_error()
    assert not lib.formhost_pool_create_mixed(None, 2, 200)
    assert not lib.formhost_pool_create_mixed(arr, 0, 200)
    traces = (C.c_void_p * 2)()
    assert not lib.formhost_batch_replay_create_mixed(traces, 2, arr, None)
    assert b"device" in lib.formhost_last_error()
    assert not lib.formhost_batch_replay_create_mixed(None, 2, arr, None)


def test_python_wrappers_check_list_lengths():
    from form_b200.pipeline import BatchReplay, EstimatorPool

    p = _capi.default_est_params(16, 1800)
    with pytest.raises(ValueError, match="2 params for 3 sequences"):
        BatchReplay([None, None, None], [p, p])
    with pytest.raises(ValueError, match="2 params for 3 sequences"):
        EstimatorPool([p, p], 3)
    with pytest.raises(TypeError, match="n_sequences"):
        EstimatorPool(p)


def test_sweep_keys_are_form_default_params():
    import form

    defaults = form.FORM.default_params()
    assert set(sweep.PARAM_FIELDS) == set(defaults)
    # every key's default lands on the field that holds the same default
    p = _capi.default_est_params(64, 1024)
    for key, value in defaults.items():
        field = sweep.PARAM_FIELDS[key][0]
        target = p.hot if field.startswith("hot.") else p
        assert getattr(target, field.split(".")[-1]) == value, key


def test_sweep_variant_parsing_and_mapping():
    assert sweep.parse_variant("form") == ("form", {})
    name, ov = sweep.parse_variant("abl:point_feats_per_sector=0, disable_smoothing=true,max_dist_map=0.25")
    assert name == "abl"
    assert ov == {"point_feats_per_sector": 0, "disable_smoothing": True, "max_dist_map": 0.25}
    p = sweep.est_params(16, 1800, ov)
    assert (p.hot.num_rows, p.hot.num_columns) == (16, 1800)
    assert p.hot.point_feats_per_sector == 0 and p.disable_smoothing == 1
    assert p.hot.min_dist_map == 0.25  # max_dist_map -> the map's min_dist_map, as FORM.set_params
    q = sweep.est_params(16, 1800, {"num_sectors": 8, "max_dist_matching": 1.0, "new_pose_threshold": 1e-3,
                                    "max_num_keyscans": 20})
    assert q.hot.num_sectors == 8 and q.hot.max_dist_matching == 1.0
    assert q.new_pose_threshold == 1e-3 and q.max_num_keyscans == 20
    assert sweep.parse_variant("off:disable_smoothing=false")[1] == {"disable_smoothing": False}


@pytest.mark.parametrize("spec, match", [
    ("x:min_dist_map=0.2", "unknown parameter 'min_dist_map'; valid keys: .*max_dist_map"),
    ("x:bogus=1", "valid keys: disable_smoothing, keyscan_match_ratio"),
    ("x:num_sectors", "not key=value"),
    ("x:num_sectors=2.5", "integer"),
    ("x:disable_smoothing=maybe", "true or false"),
    (":num_sectors=4", "name"),
    ("gt", "ground-truth"),
])
def test_sweep_rejects_bad_variants(spec, match):
    with pytest.raises(ValueError, match=match):
        sweep.parse_variant(spec)


def test_sweep_rejects_duplicate_names_and_unknown_keys_on_the_command_line(capsys):
    with pytest.raises(ValueError, match="duplicate variant name 'a'"):
        sweep.parse_variants(["a", "b:num_sectors=4", "a:num_sectors=8"])
    with pytest.raises(SystemExit):
        sweep.main(["--variant", "a:nope=1", "--scans", "1"])
    assert "valid keys" in capsys.readouterr().err
    with pytest.raises(ValueError, match="valid keys"):
        sweep.est_params(16, 1800, {"nope": 1})
