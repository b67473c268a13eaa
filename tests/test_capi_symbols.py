"""CPU: the C-ABI library loads, exports every symbol include/b200fold.h declares, and fails loudly
(never falls back) when there is no GPU.  The parameter loader is host code and is checked here too."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "b200fold.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bf_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from desirna_b200 import engine
    L = engine.lib()
    names = declared_symbols()
    assert len(names) >= 10
    for n in names:
        assert hasattr(L, n), n


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from desirna_b200 import engine
    with pytest.raises(engine.EngineError) as ei:
        engine.init(0)
    assert ei.value.code == 1  # BF_ERR_CUDA


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "desirna_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cc", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("# oracle", ""), os.path.join(dp, f)
                assert "orc_" not in txt, os.path.join(dp, f)


def test_param_loader_matches_oracle_loader(oracle):
    """bf_params.cc (product loader) against the oracle's independent parser + the constants SURVEY A.2 quotes."""
    from desirna_b200 import engine
    engine.params_builtin(1999)  # host-side parse works without a GPU
    g = engine.params_get
    assert g("stack", 1, 1) == -240
    assert [g("hairpin", k) for k in (3, 4, 5)] == [570, 560, 560]
    assert (g("MLbase"), g("MLclosing"), g("MLintern")) == (0, 340, 40)
    assert (g("DuplexInit"), g("TerminalAU"), g("ninio_m"), g("ninio_max")) == (410, 50, 50, 300)
    assert g("lxc1000") == 107856
    assert g("n_tetra") == 30 and g("n_tri") == 0 and g("n_hexa") == 0
    key = 0
    for ch in "GGGGAC":
        key = key * 4 + "ACGU".index(ch)
    assert g("tetra_e", key) == 20
    for name, dims in (("stack", (8, 8)), ("mmH", (8, 5, 5)), ("mmI", (8, 5, 5)), ("mm1nI", (8, 5, 5)), ("mm23I", (8, 5, 5)),
                       ("mmM", (8, 5, 5)), ("mmE", (8, 5, 5)), ("dangle5", (8, 5)), ("dangle3", (8, 5)), ("int11", (8, 8, 5, 5)),
                       ("int21", (8, 8, 5, 5, 5)), ("hairpin", (31,)), ("bulge", (31,)), ("interior", (31,))):
        import itertools
        for idx in itertools.product(*[range(1 if (d in (8,) and len(dims) > 1) else 0, d) for d in dims]):
            assert g(name, *idx) == oracle.get(name, *idx), (name, idx)
    # int22: sample (6^2 * 4^4 standard entries + NS fills)
    import random
    rnd = random.Random(1)
    for _ in range(3000):
        idx = (rnd.randint(1, 7), rnd.randint(1, 7)) + tuple(rnd.randint(1, 4) for _ in range(4))
        assert g("int22", *idx) == oracle.get("int22", *idx), idx


def test_set_option_refuses_unknown_keys():
    """bf_set_option sets only the switches include/b200fold.h lists; a removed or misspelt key is an error, not a no-op."""
    from desirna_b200 import engine
    L = engine.lib()
    assert L.bf_set_option(b"mfe_nw", 4) == 5  # BF_ERR_ARG
    assert L.bf_set_option(b"design_graph", 1) == 5
    assert L.bf_set_option(b"wide", 0) == 0
    assert L.bf_set_option(b"wide", -1) == 0  # back to the default rule


def test_params_2004_is_reported_unavailable():
    from desirna_b200 import engine
    with pytest.raises(engine.EngineError) as ei:
        engine.params_builtin(2004)
    assert ei.value.code == 4
