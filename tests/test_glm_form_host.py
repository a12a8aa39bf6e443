"""CPU: plumbing of the GLM evaluation-form option (b2m_model_options.glm_form) through the C ABI and the Python API."""
import ctypes
import inspect
import os
import re

import pytest

from mlx_mcmc_b200 import _cabi, engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_glm_form_is_carved_out_of_the_reserved_words():
    lib = _cabi.load()
    assert ctypes.sizeof(_cabi.ModelOptions) == lib.b2m_options_size() == 32
    assert _cabi.ModelOptions.glm_form.offset == 16 and _cabi.ModelOptions.reserved.offset == 20
    assert len(_cabi.ModelOptions().reserved) == 3
    assert _cabi.ABI_VERSION == 4 and lib.b2m_abi_version() == 4
    header = open(os.path.join(ROOT, "include", "b200mcmc.h")).read()
    assert re.search(r"B2M_FORM_AUTO = 0, B2M_FORM_STREAM = 1, B2M_FORM_GRAM = 2", header)
    assert re.search(r"int32_t glm_form;.*\n\s*int32_t reserved\[3\];", header)


def test_glm_form_names():
    assert _cabi.GLM_FORMS == {"auto": 0, "stream": 1, "gram": 2}
    assert (_cabi.FORM_AUTO, _cabi.FORM_STREAM, _cabi.FORM_GRAM) == (0, 1, 2)
    assert inspect.signature(engine.compile_model).parameters["glm_form"].default == "auto"
    assert inspect.signature(engine.DeviceModel.__init__).parameters["glm_form"].default == "auto"
    assert "b2m_model_glm_form" in _cabi.EXPORTS


def _create(opt):
    lib = _cabi.load()
    t = (_cabi.Term * 1)()
    t[0].dist = 0
    t[0].length = 1
    return lib, lib.b2m_model_create(t, 1, None, 0, None, 0, 1, ctypes.byref(opt), ctypes.byref(ctypes.c_void_p()))


@pytest.mark.parametrize("bad", [3, -1, 99])
def test_unknown_glm_form_is_refused(bad):
    opt = _cabi.ModelOptions()
    opt.glm_form = bad
    lib, rc = _create(opt)
    assert rc != 0 and b"glm_form" in lib.b2m_last_error()


@pytest.mark.parametrize("word", [0, 1, 2])
def test_reserved_words_are_still_refused(word):
    opt = _cabi.ModelOptions()
    opt.glm_form = _cabi.FORM_GRAM
    opt.reserved[word] = 1
    lib, rc = _create(opt)
    assert rc != 0 and b"reserved" in lib.b2m_last_error()


def test_model_glm_form_of_no_model():
    lib = _cabi.load()
    assert lib.b2m_model_glm_form(None) == -1

