"""The per-iteration vector kernels (iter_head / iter_mid / iter_tail) recompute in registers what they used to
store and read back (the affine and combined directions of the LP rows, lambda of an LP-only problem, the
corrected x / y directions).  Every recomputation repeats the stored value's expression with the same roundings,
so the solver's results must not move by a single bit.  This test runs three batched workloads on the CPU
emulator and compares SHA-256 digests of their results with digests recorded from the build that still stored
those rows.

The digests were produced with `python tests/test_vector_passes.py <emulator library>` from the build before the
change; the same command prints them for the current build.  Each digest covers the float64 bytes of one output
over the whole batch (exit flags, iteration and refinement counts converted to float64)."""
import hashlib
import os
import sys

import numpy as np
import pytest

KEYS = ("x", "y", "z", "s", "exit", "iter", "nitref1", "nitref2", "nitref3")

# workload -> output -> sha256 of its float64 bytes, recorded from the build that stored the rows
DIGESTS = {
    'MPC02x64': {
        'x': '4043f678c3255d82e5b85fe15ef0754e963e2917755489056a60301cd157c309',
        'y': '346d7a20fed16a839999f65adc9479e62a04061f64dedf598a312fbb0d26dbe3',
        'z': '6fb5c78cdc2b9722d07265989d4878f4e3eb462080843131dc5164c5085940b1',
        's': '469fd79b90c0ae92eb4800906f0e859f142e80fe119a5462772d8f7f0326315c',
        'exit': '076a27c79e5ace2a3d47f9dd2e83e4ff6ea8872b3c2218f66c92b89b55f36560',
        'iter': 'b64f2c9679e65d294d60765ce6f584f3013a6a048e9d14c2497112bedb1dc545',
        'nitref1': 'e31bedb0d9a84d336f4601611ba5c1f0c14a22ede9bbb52afb09092dc79d6b67',
        'nitref2': 'e31bedb0d9a84d336f4601611ba5c1f0c14a22ede9bbb52afb09092dc79d6b67',
        'nitref3': '076a27c79e5ace2a3d47f9dd2e83e4ff6ea8872b3c2218f66c92b89b55f36560',
    },
    'socmpc_x32': {
        'x': 'd14152fd946f4e76ed382f82ad8d58985dd0ea0e2f5a281add2679ebf9f51ee4',
        'y': 'aca16cc3b417f35217056ec9023e68c762d4609faf70fd9f611e4bf270f0fb5e',
        'z': '6426b30872d1e0044c8e3db873140d662d05a3e700f79941cd854f47fd4cdd74',
        's': '9d6c23df2a88d31265476c6ac1750f85692ec5a9341de2d66fb66a98f589db17',
        'exit': '5341e6b2646979a70e57653007a1f310169421ec9bdd9f1a5648f75ade005af1',
        'iter': '570d340ee68766f5ccedebe6e30ee5575345e714f7a707e60a3875b9376bdac7',
        'nitref1': 'acfc7c36fce590b14adfc8a479e0dcd297e910a7212694c976c8b4284d34c144',
        'nitref2': 'acfc7c36fce590b14adfc8a479e0dcd297e910a7212694c976c8b4284d34c144',
        'nitref3': 'f89073db4358a04ce6582b3ab9bf183179a637156193efd5518d611568c0be7f',
    },
    'lp_afiro_x16': {
        'x': '8744ad12aee4f4dbc36687a8ecd1fee2469502f71812c477869d32ca3f8fa24d',
        'y': '5fcd6c0925052ad0be89276d4ec9c4036c71e484723ab884ce25db66818218a5',
        'z': '7501ffefa63e24ff4aad1caa26e07f4518c86ff348d575637556acac1692e236',
        's': '2cce3d9441611dedeb158bca7ddfd29beb4f9dc6b4f97666f496d70b58d553a9',
        'exit': '38723a2e5e8a17aa7950dc008209944e898f69a7bd10a23c839d341e935fd5ca',
        'iter': '0e779f6ba09500d6509beebb543d4b31df403e9c0227e5fb3801ea61d6cfccdb',
        'nitref1': 'dbd8ebb4d364765882694170cedf5afc7702dd5338a7198705c45b613f6e1c9d',
        'nitref2': 'dbd8ebb4d364765882694170cedf5afc7702dd5338a7198705c45b613f6e1c9d',
        'nitref3': '38723a2e5e8a17aa7950dc008209944e898f69a7bd10a23c839d341e935fd5ca',
    },
}


def _cases():
    import oracle
    from eicos_b200.workloads import perturbed, soc_mpc, soc_mpc_batch
    P = oracle.load_fixture("MPC02")
    yield "MPC02x64", P, perturbed(P, 64, rel={"h": 0.002, "b": 0.02}, seed=5)
    P = soc_mpc(T=12)
    yield "socmpc_x32", P, soc_mpc_batch(P, 32)
    P = oracle.load_fixture("lp_afiro")
    yield "lp_afiro_x16", P, perturbed(P, 16, rel=0.02, seed=5)


def _digests(lib, P, W):
    from eicos_b200.binding import BatchSolver
    batch = W["hs"].shape[0]
    # one instance per tile in the emulator: 3 workers split the rows unevenly, and the batch is large enough
    # for active-set compaction to move instances between the head and the rest of an iteration
    out = BatchSolver(P, lib=lib, capacity=batch, workers=3).solve(batch, hs=W["hs"], bs=W["bs"])
    for k in ("nitref1", "nitref2", "nitref3"):
        out[k] = np.array([i[k] for i in out["info"]])
    return {k: hashlib.sha256(np.ascontiguousarray(out[k], dtype=np.float64).tobytes()).hexdigest() for k in KEYS}


@pytest.mark.parametrize("name", ["MPC02x64", "socmpc_x32", "lp_afiro_x16"])
def test_results_are_bit_identical(emu_lib, name):
    for case, P, W in _cases():
        if case == name:
            assert _digests(emu_lib, P, W) == DIGESTS[name]


if __name__ == "__main__":
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, ROOT)
    from eicos_b200.binding import Library
    lib = Library(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "emu", "_build", "libeicos_emu.so"))
    for case, P, W in _cases():
        print(f"    {case!r}: {{")
        for k, v in _digests(lib, P, W).items():
            print(f"        {k!r}: {v!r},")
        print("    },")
