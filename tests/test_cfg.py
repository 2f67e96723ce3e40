"""Classifier-free guidance (UbConfig.class_dropout) without a GPU: the parameter layout of a guided model (exactly a
(K + 1)-class model), the configs the library refuses, and the new config field's place in the C struct and in the
Python mirror."""
import math
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CONFIGS = [
    dict(num_classes=10),
    dict(num_classes=1, H=32, W=32, channel_mult=(1, 2)),
    dict(num_classes=10, learn_sigma=1),
    dict(num_classes=1000, learn_sigma=1, use_scale_shift_norm=1, resblock_updown=1, head_size=64, C_model=128),
    dict(num_classes=5, super_res=4, noise_schedule=1, dropout=0.1),
]


@pytest.mark.parametrize("kw", CONFIGS, ids=[str(i) for i in range(len(CONFIGS))])
@pytest.mark.parametrize("p", [0.1, 0.5, 1e-6])
def test_num_params_is_that_of_one_more_class(ub, kw, p):
    K = kw["num_classes"]
    cfg = ub.default_config(**kw, class_dropout=p)
    plus = ub.default_config(**{**kw, "num_classes": K + 1})
    n = ub.num_params(cfg)
    assert n > 0 and n == ub.num_params(plus)
    assert n == ub.num_params(ub.default_config(**kw)) + 4 * cfg.C_model  # one label row of 4 * C_model


@pytest.mark.parametrize("kw", CONFIGS, ids=[str(i) for i in range(len(CONFIGS))])
def test_zero_dropout_leaves_the_model_unchanged(ub, kw):
    assert ub.default_config().class_dropout == 0.0
    assert ub.num_params(ub.default_config(**kw, class_dropout=0.0)) == ub.num_params(ub.default_config(**kw))


@pytest.mark.parametrize("p", [-0.1, 1.0, 1.5, math.nan, math.inf, -math.inf])
def test_refused_dropout_rates(ub, p):
    assert ub.num_params(ub.default_config(num_classes=10, class_dropout=p)) == 0
    assert b"class_dropout must lie in [0, 1) and needs num_classes > 0" in ub.lib().ub_last_error()


def test_dropout_needs_classes(ub):
    assert ub.num_params(ub.default_config(class_dropout=0.1)) == 0
    err = ub.lib().ub_last_error()
    assert b"needs num_classes > 0" in err and b"num_classes = 0" in err
    with pytest.raises(ub.UbError, match="class_dropout"):
        ub.Trainer(B=2, class_dropout=0.1)  # refused before any device work


def _header_fields():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "unet_b200.h")).read(), flags=re.S)
    body = re.search(r"typedef struct \{([^{}]*)\} UbConfig;", src).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            for part in decl.split(","):
                names.append(re.sub(r"\[.*\]", "", part.split()[-1]).lstrip("*"))
    return names


def test_class_dropout_is_the_last_field(ub):
    names = _header_fields()
    assert names[-1] == "class_dropout"
    assert [f[0] for f in ub.UbConfig._fields_] == names  # the Python mirror follows the header
    assert ub.UbConfig.class_dropout.offset == ub.UbConfig.noise_schedule.offset + 4
    assert ub.UbConfig.class_dropout.size == 4


def test_new_entry_points_are_declared(ub):
    L = ub.lib()
    for name in ("ub_trainer_set_guidance", "ub_trainer_get_effective_labels"):
        assert hasattr(L, name), name
