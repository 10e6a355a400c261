"""The live-NEE k_shade instantiations run 4 CTAs of 160 threads per SM (SHADE_THREADS_NEE): that shape needs them at <= 96
registers WITHOUT spills, which the phase structure of the trip is what provides.  Checked on the built engine.o (no GPU)."""
import importlib.util
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tool():
    spec = importlib.util.spec_from_file_location("shade_regs", os.path.join(ROOT, "tools", "shade_regs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_live_nee_shade_fits_its_shape_without_spills():
    rows = {name: (reg, stack, st, ld) for name, reg, stack, st, ld in _tool().table()}
    nee = [n for n in rows if n.startswith("k_shade<1,") and n.endswith("true, 160, false>")]
    assert len(nee) == 5, sorted(rows)
    for n in nee:
        reg, stack, st, ld = rows[n]
        assert reg <= 96 and stack == 0 and st == 0 and ld == 0, (n, rows[n])
    # the dead-MIS kernels keep 2 CTAs of 256 threads; at that bound they must not spill more than they used to (134 bytes)
    for n in (n for n in rows if n.startswith("k_shade<2, 5,") and ", true, 256, false>" in n):
        assert rows[n][2] <= 134, (n, rows[n])
