"""The C++ host mirror (include/gl_plonky2.hpp: PolynomialBatch / MerkleTree / Challenger / fri_proof / prove_openings with
upstream's names and panics) compiled into tests/cpp/build/host_mirror_test, which checks it against the C oracle.

CPU: the header compiles warning-free against include/gl_commit.h, links the product library, and refuses to run without a
device (no CPU fallback).  GPU: the whole binary — commits, Merkle paths under the verifier's rule, the FRI commit phase,
proof of work and query rounds on the oracle's transcript, and the golden openings fixture."""
import json
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "host_mirror_test.cpp")
OUT_DIR = os.path.join(ROOT, "tests", "cpp", "build")
BIN = os.path.join(OUT_DIR, "host_mirror_test")


def build_host_mirror_test() -> str:
    import plonky25_b200 as g
    from oracle_c import build_oracle
    lib = g.build()
    ora = build_oracle()
    deps = [SRC, os.path.join(ROOT, "include", "gl_plonky2.hpp"), os.path.join(ROOT, "include", "gl_commit.h"), lib, ora]
    if os.path.exists(BIN) and all(os.path.getmtime(d) <= os.path.getmtime(BIN) for d in deps):
        return BIN
    os.makedirs(OUT_DIR, exist_ok=True)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), SRC, "-o", BIN,
           "-L", os.path.dirname(lib), "-lgl_commit", "-L", os.path.dirname(ora), "-lgl_oracle",
           "-Wl,-rpath,$ORIGIN/../../../plonky2.5_b200", "-Wl,-rpath,$ORIGIN/../../../oracle", "-pthread"]
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run(cmd, check=True, env=env)
    return BIN


def build_host_mirror_test_double() -> str:
    """the same test source linked against tests/cpp/abi_test_double.cpp (the C ABI restated over the oracle; test infrastructure):
    exercises the host logic of the C++ mirror and of the test itself without a device"""
    from oracle_c import build_oracle
    ora = build_oracle()
    exe = BIN + "_double"
    dbl = os.path.join(ROOT, "tests", "cpp", "abi_test_double.cpp")
    deps = [SRC, dbl, os.path.join(ROOT, "include", "gl_plonky2.hpp"), os.path.join(ROOT, "include", "gl_commit.h"), ora]
    if os.path.exists(exe) and all(os.path.getmtime(d) <= os.path.getmtime(exe) for d in deps):
        return exe
    os.makedirs(OUT_DIR, exist_ok=True)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), SRC, dbl, "-o", exe,
                    "-L", os.path.dirname(ora), "-lgl_oracle", "-Wl,-rpath,$ORIGIN/../../../oracle", "-pthread"], check=True, env=env)
    return exe


def _flatten_golden(path: str) -> None:
    """tests/golden/openings_fri.json as 'key v v v ...' lines for the C++ reader"""
    f = json.load(open(os.path.join(ROOT, "tests", "golden", "openings_fri.json")))
    assert [len(b["polynomials"]) for b in f["batches"]] == [sum(f["widths"]), 2]     # the instance shape the binary rebuilds
    lines = {k: f[k] if isinstance(f[k], list) else [f[k]]
             for k in ("log_n", "widths", "rate_bits", "cap_height", "arity_bits", "pow_bits", "col_seeds", "transcript_prefix", "alpha",
                       "fri_final_poly", "pow_witness", "query_indices")}
    lines["commit_phase_caps"] = [x for cap in f["commit_phase_caps"] for x in cap]
    lines["fri_final_poly"] = [x for e in f["fri_final_poly"] for x in e]
    lines["point0"], lines["point1"] = f["batches"][0]["point"], f["batches"][1]["point"]
    with open(path, "w") as out:
        for k, v in lines.items():
            out.write(k + " " + " ".join(str(int(x)) for x in v) + "\n")


def _device_present() -> bool:
    """what the binaries themselves see: CUDA's device count (a GPU's device node need not be /dev/nvidia0, e.g. in a container
    that is given one GPU of a larger machine)"""
    import plonky25_b200 as g
    return g._lib.load().gl_device_count() > 0


def test_cpp_host_mirror_compiles_and_has_no_cpu_path():
    exe = build_host_mirror_test()
    if _device_present():
        pytest.skip("GPU present")
    r = subprocess.run([exe, "--expect-no-device"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout


def test_cpp_header_is_self_contained(tmp_path):
    """include/gl_plonky2.hpp compiles on its own (C++17, no torch / CUDA headers needed by a host that binds it)"""
    tu = tmp_path / "tu.cpp"
    tu.write_text('#include "gl_plonky2.hpp"\nint main() { plonky2::FriParams p; return int(p.lde_bits()); }\n')
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(tu)],
                   check=True, env=env)


def test_cpp_host_mirror_host_logic_on_abi_double(tmp_path):
    """handle lifetimes, transcript order, query-round assembly and panic mapping of include/gl_plonky2.hpp, device-free"""
    exe = build_host_mirror_test_double()
    gold = tmp_path / "openings_fri.txt"
    _flatten_golden(str(gold))
    r = subprocess.run([exe, "--golden", str(gold)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]
    # the product library is not part of that binary, and the product never links the double
    ldd = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "libgl_commit" not in ldd
    nm = subprocess.run(["nm", "-D", "--undefined-only", os.path.join(ROOT, "plonky2.5_b200", "libgl_commit.so")], capture_output=True, text=True).stdout
    assert "glo_" not in nm, "libgl_commit.so must not reference the oracle"


def test_cpp_host_mirror_under_sanitizers(tmp_path):
    """the header's host logic (handle ownership, moves, query-round assembly) under AddressSanitizer + UBSan + LeakSanitizer, on the
    ABI double: every device handle a mirror object owns must be released exactly once"""
    from oracle_c import build_oracle
    ora = build_oracle()
    exe = str(tmp_path / "host_mirror_asan")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    r = subprocess.run([cxx, "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-I", os.path.join(ROOT, "include"),
                        SRC, os.path.join(ROOT, "tests", "cpp", "abi_test_double.cpp"), "-o", exe, "-L", os.path.dirname(ora), "-lgl_oracle",
                        "-Wl,-rpath," + os.path.dirname(ora), "-pthread"], capture_output=True, text=True, env=env)
    if r.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + r.stderr[-300:])
    gold = tmp_path / "openings_fri.txt"
    _flatten_golden(str(gold))
    env["ASAN_OPTIONS"] = "detect_leaks=1"
    r = subprocess.run([exe, "--golden", str(gold)], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "ALL OK" in r.stdout and "ERROR" not in r.stderr and "runtime error" not in r.stderr, r.stdout[-2000:] + r.stderr[-4000:]


def _cxx(args):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), *args], check=True, env=env)


def build_cpp_tools() -> dict:
    """tools/cbench.cpp (e2e through the C ABI from C++) and tests/cpp/variant_bench.cpp (parity + timing of library variants)"""
    import plonky25_b200 as g
    from oracle_c import build_oracle
    lib, ora = g.build(), build_oracle()
    os.makedirs(OUT_DIR, exist_ok=True)
    out = {"cbench": os.path.join(OUT_DIR, "cbench"), "variant_bench": os.path.join(OUT_DIR, "variant_bench"),
           "devbench": os.path.join(OUT_DIR, "devbench"), "gates_mirror_test": os.path.join(OUT_DIR, "gates_mirror_test")}
    hdr = os.path.join(ROOT, "include", "gl_commit.h")

    def stale(exe, deps):
        return not os.path.exists(exe) or any(os.path.getmtime(d) > os.path.getmtime(exe) for d in deps)

    src = os.path.join(ROOT, "tools", "cbench.cpp")
    if stale(out["cbench"], [src, hdr, lib]):
        _cxx([src, "-o", out["cbench"], "-L", os.path.dirname(lib), "-lgl_commit", "-Wl,-rpath,$ORIGIN/../../../plonky2.5_b200", "-pthread"])
    src = os.path.join(ROOT, "tests", "cpp", "gates_mirror_test.cpp")
    if stale(out["gates_mirror_test"], [src, hdr, os.path.join(ROOT, "include", "gl_plonky2.hpp"), lib]):
        _cxx([src, "-o", out["gates_mirror_test"], "-L", os.path.dirname(lib), "-lgl_commit", "-Wl,-rpath,$ORIGIN/../../../plonky2.5_b200", "-pthread"])
    src = os.path.join(ROOT, "tools", "devbench.cpp")
    if stale(out["devbench"], [src, hdr, lib]):
        _cxx([src, "-o", out["devbench"], "-L", os.path.dirname(lib), "-lgl_commit", "-Wl,-rpath,$ORIGIN/../../../plonky2.5_b200", "-pthread"])
    src = os.path.join(ROOT, "tests", "cpp", "variant_bench.cpp")
    if stale(out["variant_bench"], [src, hdr, ora]):
        _cxx([src, "-o", out["variant_bench"], "-L", os.path.dirname(ora), "-lgl_oracle", "-Wl,-rpath,$ORIGIN/../../../oracle", "-ldl", "-pthread"])
    return out


def test_cpp_tools_build_and_refuse_to_run_without_a_device():
    exe = build_cpp_tools()
    if _device_present():
        pytest.skip("GPU present")
    r = subprocess.run([exe["cbench"]], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "no CPU fallback" in r.stdout
    r = subprocess.run([exe["variant_bench"], "--log-n", "8", os.path.join(ROOT, "plonky2.5_b200", "libgl_commit.so")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "no CPU fallback" in r.stdout


@pytest.mark.gpu
def test_cpp_tools_on_gpu():
    """cbench: copy-back (pinned) equals the resident batch; variant_bench: the product library is parity-green through dlopen"""
    exe = build_cpp_tools()
    r = subprocess.run([exe["cbench"], "12", "20", "1", "2", "1", "14", "135", "3", "4", "2"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.count("copy-back == gl_tree_read of the resident batch") == 2, r.stdout[-3000:]
    r = subprocess.run([exe["variant_bench"], "--log-n", "14", os.path.join(ROOT, "plonky2.5_b200", "libgl_commit.so")],
                       capture_output=True, text=True, timeout=300)
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert r.returncode == 0 and line["parity_2p10x135"] and line["parity_noncanonical"] and line["parity_2p12x9"], r.stdout[-3000:]


@pytest.mark.gpu
def test_cpp_host_mirror_matches_oracle_on_gpu(tmp_path):
    exe = build_host_mirror_test()
    gold = tmp_path / "openings_fri.txt"
    _flatten_golden(str(gold))
    r = subprocess.run([exe, "--golden", str(gold)], capture_output=True, text=True, timeout=600)
    print(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert "ALL OK" in r.stdout


@pytest.mark.gpu
def test_cpp_gates_mirror_on_gpu():
    """QuotientAccumulator / partial_products_and_zs / poseidon2_gate_witness of include/gl_plonky2.hpp against their own identities"""
    exe = build_cpp_tools()["gates_mirror_test"]
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
