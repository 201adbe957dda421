"""Generates tests/golden/rustc_hash_k_windows.npz: the machine code around rustc-hash 2.x's multiplier K in compiled
Rust extension modules that link it (tiktoken, tokenizers, outlines_core, wherever they are installed), the evidence
tests/test_oracle_kats.py::test_fxhasher_constants_against_compiled_rustc_hash reads for K and the rotate of `finish()`.

Every occurrence of K (a 64-bit immediate, little endian) is stored with the 88 bytes that follow it: `windows` is
uint8 [N, 96], `sources` names the module file and version of each row.
"""
import glob
import importlib.metadata
import importlib.util
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
K = bytes.fromhex("c5a9622eea7a35f1")           # 0xf1357aea2e62a9c5, little endian
WINDOW = 96


def main():
    windows, sources = [], []
    for mod in ("tiktoken", "tokenizers", "outlines_core"):
        spec = importlib.util.find_spec(mod)
        if not (spec and spec.submodule_search_locations):
            continue
        version = importlib.metadata.version(mod.replace("_", "-"))
        for d in spec.submodule_search_locations:
            for f in sorted(glob.glob(d + "/*.so")):
                data = open(f, "rb").read()
                i = data.find(K)
                while i >= 0:
                    windows.append(np.frombuffer(data[i:i + WINDOW].ljust(WINDOW, b"\0"), dtype=np.uint8))
                    sources.append(f"{mod} {version}: {os.path.basename(f)}")
                    i = data.find(K, i + 8)
    np.savez_compressed(os.path.join(HERE, "rustc_hash_k_windows.npz"), windows=np.stack(windows), sources=np.array(sources))
    print(len(windows), "windows from", sorted(set(sources)))


if __name__ == "__main__":
    main()
