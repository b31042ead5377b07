"""Shows that the GEMM mode tests (tests/test_gpu_gemm_modes.py) have teeth: breaks one rule of the NumPy model at a
time, reruns every call-site case and the tile-subset and m_dec checks against the unchanged kernel on the GPU, and
reports which checks fail.  Every mutation must be caught by at least one check; the kernel itself is never changed.

    python scripts/gemm_model_mutations.py
"""
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MUTATIONS = {  # name: (text in the model, replacement)
    "drop the b_tri trim": ("ke = min(ke, (j0 // TB + 1) * TB)", "pass"),
    "drop the a_tri = 1 trim": ("kb = i0 + a_off\n", "kb = 0\n"),
    "a_tri = 2 trim ignores a_row_off": ("ke = i0 + a_off + BM", "ke = i0 + BM"),
    "Adiag tile index without a_row_off": ("tia = ti + a_off // TB", "tia = ti"),
    "no Bdiag redirect": ('if "Bdiag" in d and k0 // TB == jb:', "if False:"),
    "Adiag not advanced per problem": ('b, o = ptr("Adiag", q)', 'b, o = d["Adiag"]'),
    "split-K chunk not clipped to the k-range": (
        'kb, ke = max(kb, chunk * d["klen"]), min(ke, (chunk + 1) * d["klen"])',
        'kb, ke = chunk * d["klen"], (chunk + 1) * d["klen"]'),
    "C advanced per problem, not per entry": ('bC, oC = ptr("C", qe)', 'bC, oC = ptr("C", q)'),
    "s_row_off ignored": ('a_off = d.get("a_row_off", 0) + q * d.get("s_row_off", 0)', 'a_off = d.get("a_row_off", 0)'),
    "no m_dec exit": ('if i0 >= M - q * d.get("m_dec", 0):', "if i0 >= M:"),
    "beta = 0 reads C": ("if beta != 0.0:", "if True:"),
    "no transposed store": ('if "Ct" in d:', "if False:"),
    "lower_only rows of 2 ti + 1 tiles": ("out.append((t, L - t * (t + 1)))", "out.append((t, min(L - t * (t + 1), 2 * t)))"),
    "tile subset starts at 0": ("range(first, tiles, stride)", "range(0, tiles, stride)"),
}


def load(src):
    mod = types.ModuleType("gemm_modes_mutant")
    mod.__file__ = os.path.join(ROOT, "tests", "test_gpu_gemm_modes.py")
    exec(compile(src, mod.__file__, "exec"), mod.__dict__)
    return mod


def checks(m):
    import zlib

    out = {}
    for name in sorted(m.CASES):
        d, lens = m.CASES[name]()
        out[name] = lambda d=d, lens=lens, name=name: m.run_case(d, lens, seed=zlib.crc32(name.encode()))
    out["tile_subsets_world3"] = lambda: m.test_uut_tile_subsets_partition_lower_only(3)
    out["m_dec_tail"] = m.test_m_dec_tail_untouched
    return out


def main():
    src = open(os.path.join(ROOT, "tests", "test_gpu_gemm_modes.py")).read()
    base = checks(load(src))
    for name, fn in base.items():
        fn()  # the unchanged model passes everything
    print(f"unchanged model: all {len(base)} checks pass")
    missed = []
    for label, (old, new) in MUTATIONS.items():
        assert src.count(old) == 1, label
        failed = []
        for name, fn in checks(load(src.replace(old, new))).items():
            try:
                fn()
            except (AssertionError, IndexError, ValueError):
                failed.append(name)
        print(f"{label:45s} caught by {len(failed):2d}: {', '.join(failed)}")
        if not failed:
            missed.append(label)
    if missed:
        print("NOT CAUGHT:", missed)
        sys.exit(1)
    print(f"all {len(MUTATIONS)} mutations caught")


if __name__ == "__main__":
    main()
