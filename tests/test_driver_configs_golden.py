"""CPU: the drivers' MODEL_CONFIG / TRAIN_CONFIG / RANDOM_SEED_LIST against the reference drivers' hyper-parameters
recorded in the golden fixtures' metadata (tests/golden/make_golden.py CASES, make_golden_yahoo.py CFG, each citing
the reference driver lines it was taken from).  No reference checkout needed; test_ref_loaders_evaluators.py compares
the full config dictionaries and the item-pool flags with the live reference sources where a checkout is present."""
import importlib
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
COEF = {"lr": "lr", "c_inv": "invariant_coe", "c_ea": "env_aware_coe", "c_env": "env_coe", "c_L2": "L2_coe",
        "c_L1": "L1_coe"}

# fixture -> (driver, meta keys that are the driver's own values).  Batch sizes of the scaled-down fixtures are not
# the driver's; implicit_k6 turns reg_only_embed off on purpose (the classifier is regularised too).
CASES = {
    "coat_explicit": ("Coat_InvPref_explicit", ("K", "D", "B", "roe", "ree", "alpha", "crw", "rrw", "seed", *COEF)),
    "yahoo_explicit_full": ("Yahoo_InvPref_explicit", ("K", "D", "B", "roe", "ree", "crw", "rrw", "seed", *COEF)),
    "explicit_sched_k5": ("Yahoo_InvPref_explicit", ("K", "D", "roe", "ree", "alpha", "crw", "rrw", "seed", *COEF)),
    "implicit_k2": ("MovieLens_InvPref", ("K", "D", "roe", "ree", "alpha", "crw", "rrw", "seed", *COEF)),
    "implicit_k6": ("MIND_InvPref", ("K", "D", "ree", "alpha", "crw", "rrw", "seed", *COEF)),
}


def _driver_value(drv, key):
    m, t = drv.MODEL_CONFIG, drv.TRAIN_CONFIG
    return {"K": m["env_num"], "D": m["factor_num"], "B": t["batch_size"], "roe": m["reg_only_embed"],
            "ree": m["reg_env_embed"], "alpha": t["alpha"], "crw": t["use_class_re_weight"],
            "rrw": t["use_recommend_re_weight"]}.get(key, t.get(COEF.get(key)))


@pytest.mark.parametrize("fixture", sorted(CASES))
def test_driver_config_matches_the_reference_values_in_the_fixture(fixture):
    name, keys = CASES[fixture]
    drv = importlib.import_module("invpref_kdd_2022_b200.drivers." + name)
    z = np.load(os.path.join(HERE, "golden", fixture + ".npz"))
    meta = dict(zip(z["meta_keys"].tolist(), z["meta_vals"].tolist()))
    for k in keys:
        if k == "seed":
            assert int(meta[k]) in drv.RANDOM_SEED_LIST, (name, meta[k])
        else:
            assert str(_driver_value(drv, k)) == meta[k], (name, k, _driver_value(drv, k), meta[k])
