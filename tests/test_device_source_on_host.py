"""The sweep kernels' own source, run on the host, against the mirror (CPU suite).

`csrc/sweep_rows.cuh` is the kernel behind BASELINE configs 2 and 3.  Its GPU parity tests need
a B200; this one needs none: tests/host_emulation/ runs the kernel source itself one OS thread
per CUDA thread (thread indices, __syncthreads, shared memory, atomics stand-ins) and the result
is compared bit for bit with oracle/msc_mirror.c, the scalar restatement every GPU parity test
uses.  What is covered here and nowhere else on the CPU: the row geometry of the walk (units,
tiles, wrap-around rows, parities), the Philox rounds shared between the words of a site, the
multiply-add forms of the class select and of the tie compare, the vertical counters of the
accumulating phase with their block reduction, in every instantiation the launcher can choose
(2D / 3D, uniform / +-J, 1 / 2 / 4 words per thread, one row or several per unit, the
256-thread and the 128-thread shape).  `k_sweep_general` of csrc/sweep_general.cu - config 4 and
every graph that is not a torus - gets the same treatment: uniform and per-replica inverse
temperatures (tempering), the degree-specialised and the run-time-degree kernels, 5 / 6 / 7
planes, 7 / 10 Philox rounds; and `k_strip_phase` of csrc/strip.cu - config 5, one lattice
bit-packed along x - as one strip and as two strips that exchange their ghost rows; and the
kernels of csrc/state_io.cu: the Philox initial state, bool <-> packed in both spin layouts, and
`k_replay`, the replay of the reference algorithm's own (site, uniform) trace, against
oracle/ising_oracle.c; `k_edge_general` of csrc/moves.cu, the bit-sliced two-spin edge moves; and
the other checkerboard kernels: one launch per colour phase (non-default planes / rounds, per-replica
betas), the cooperative chunk behind a grid barrier, the thread-block-cluster chunk that small
lattices run (with per-sweep energies, with per-replica betas, with the satisfied-bond counts of
the last sweep that a tempering cycle reads), and the count-only pass.  With `k_pt_cycle` of
csrc/pt_device.cu on top, a whole tempering run - chunks of sweeps, energies, time averages, swap
decisions, slot maps, rebuilt threshold tables, slot-ordered samples - is replayed on the host as
ising_pt_timesteps_sample enqueues it and compared with the mirror's.
The library itself is not involved and stays CUDA-only.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pyisingmontecarlo_b200", "csrc")
EMU = os.path.join(ROOT, "tests", "host_emulation")


def _cut(text, start_marker, end_marker=None, what=""):
    """text without [start_marker, end_marker) (to the end when end_marker is None); both must exist"""
    i = text.find(start_marker)
    assert i >= 0, f"marker not found ({what}): {start_marker!r}"
    if end_marker is None:
        return text[:i]
    k = text.find(end_marker, i)
    assert k >= 0, f"marker not found ({what}): {end_marker!r}"
    return text[:i] + text[k:]


def prepare_sources(dst):
    """Copies of the device headers with what only nvcc can digest taken out.  Every edit is an
    exact, asserted text operation, so a change of the source that the emulation does not follow
    fails here instead of testing something else."""
    os.makedirs(dst, exist_ok=True)
    for name in ("kernels.h", "philox.h"):
        with open(os.path.join(CSRC, name)) as f, open(os.path.join(dst, name), "w") as g:
            g.write(f.read())

    msc = open(os.path.join(CSRC, "msc_device.cuh")).read()
    line = "#include <cooperative_groups.h>\n"               # cuda_on_host.h stands in for what is used of it
    assert msc.count(line) == 1 and msc.count("namespace cg = cooperative_groups;\n") == 1
    msc = msc.replace(line, "")
    inc = '#include "../../include/ising_b200.h"'
    assert msc.count(inc) == 1
    msc = msc.replace(inc, '#include "%s"' % os.path.join(ROOT, "include", "ising_b200.h"))
    # the launch helpers call cudaLaunchKernelEx
    msc = _cut(msc, "// Launch with programmatic stream serialisation", "static inline uint32_t pow2_ceil",
               "launch helpers of msc_device.cuh")
    assert "__shared__" not in msc
    open(os.path.join(dst, "msc_device.cuh"), "w").write(msc)

    rows = open(os.path.join(CSRC, "sweep_rows.cuh")).read()
    # the TMA-staged variant (opt-in, mbarrier / cp.async.bulk PTX) is not emulated
    tma = ("// ------------------------------------------------------------------------------------------\n"
           "// The same colour phase with the neighbour rows staged in shared memory by the TMA unit")
    rows = _cut(rows, tma, None, "TMA variant of sweep_rows.cuh") + "\n}  // namespace ising\n"
    # programmatic dependent launch orders kernels on a stream; the emulation runs them in order
    for ptx in ('    asm volatile("griddepcontrol.launch_dependents;");\n',
                '            asm volatile("griddepcontrol.wait;" ::: "memory");\n'):
        assert rows.count(ptx) == 1, ptx
        rows = rows.replace(ptx, "")
    assert "asm" not in re.sub(r"//.*", "", rows)
    dyn = "    extern __shared__ uint32_t sm[];\n"
    assert rows.count(dyn) == 2
    rows = rows.replace(dyn, "    uint32_t* sm = emu::dyn_smem;\n")
    assert rows.count("__shared__") == 1          # s_desc, the row geometry of a chunk of units
    rows = rows.replace("__shared__", "EMU_SHARED")
    open(os.path.join(dst, "sweep_rows.cuh"), "w").write(rows)

    gen = open(os.path.join(CSRC, "sweep_general.cu")).read()
    gen = _cut(gen, "template <int K, int ROUNDS, int DEG, int V>\nstatic void gen_launch(", None,
               "launchers and other kernels of sweep_general.cu") + "\n}  // namespace ising\n"
    # dependent-launch control and the L2 prefetches of the graph arrays in front of the wait
    gen = _cut(gen, '    asm volatile("griddepcontrol.launch_dependents;");\n', "    // block = (wx lanes over replica word groups",
               "PTX preamble of k_sweep_general")
    assert "asm" not in re.sub(r"//.*", "", gen) and "__shared__" not in gen and "__syncthreads" not in gen
    assert gen.count("__global__") == 1
    open(os.path.join(dst, "sweep_general_kernel.cuh"), "w").write(gen)

    strip = open(os.path.join(CSRC, "strip.cu")).read()
    strip = _cut(strip, "template <int V>\nstatic int strip_phase_dispatch(", None,
                 "launchers and other kernels of strip.cu") + "\n}  // namespace ising\n"
    for ptx in ('    asm volatile("griddepcontrol.launch_dependents;");\n',
                '    asm volatile("griddepcontrol.wait;" ::: "memory");\n'):
        assert strip.count(ptx) == 1, ptx
        strip = strip.replace(ptx, "")
    assert "asm" not in re.sub(r"//.*", "", strip) and "__shared__" not in strip and strip.count("__global__") == 1
    open(os.path.join(dst, "strip_phase_kernel.cuh"), "w").write(strip)
    aux = open(os.path.join(CSRC, "strip.cu")).read()
    i = aux.find("__global__ void k_strip_init_random(")
    assert i >= 0
    aux, nwrap = re.subn(r"\nint launch_\w+\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", aux[i:])
    assert nwrap == 3 and "<<<" not in aux and aux.count("__global__") == 3, nwrap
    open(os.path.join(dst, "strip_aux_kernels.cuh"), "w").write("namespace ising {\n" + aux)
    fu = open(os.path.join(CSRC, "strip.cu")).read()
    i = fu.find("template <int K, int ROUNDS, int V>\n__global__ void __launch_bounds__(256, 3)\nk_strip_sweep_fused(")
    k = fu.find("// The same pass with every row staged in shared memory by the TMA unit")
    assert 0 <= i < k
    fu = fu[i:k]
    ring = "    extern __shared__ uint32_t ring_all[];"
    assert fu.count(ring) == 1 and fu.count("__shared__") == 1 and "asm" not in re.sub(r"//.*", "", fu)
    open(os.path.join(dst, "strip_fused_kernel.cuh"), "w").write(
        "namespace ising {\n" + fu.replace(ring, "    uint32_t* ring_all = emu::dyn_smem;") + "\n}  // namespace ising\n")

    io = open(os.path.join(CSRC, "state_io.cu")).read()
    # the host-side wrappers (<<< >>> launches, the SM-count query) go; the kernels stay as they are
    io, nwrap = re.subn(r"\n(?:int launch_\w+|unsigned device_sms)\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", io)
    assert nwrap == 8 and "<<<" not in io and "cudaGetDevice" not in io, nwrap
    assert io.count("__global__") == 7
    open(os.path.join(dst, "state_io_kernels.cuh"), "w").write(io)

    mv = open(os.path.join(CSRC, "moves.cu")).read()
    head = ("// ------------------------------------------------------------------------------------------\n"
            "// Edge moves on graphs whose couplings all have the same magnitude")
    i = mv.find(head)
    k = mv.find("template <int K, int ROUNDS, int DEG>\nstatic int edge_general_launch(")
    assert 0 <= i < k
    mv = '#include "msc_device.cuh"\nnamespace ising {\n' + mv[i:k] + "\n}  // namespace ising\n"
    for ptx in ('    asm volatile("griddepcontrol.launch_dependents;");\n',
                '    asm volatile("griddepcontrol.wait;" ::: "memory");\n'):
        assert mv.count(ptx) == 1, ptx
        mv = mv.replace(ptx, "")
    assert "asm" not in re.sub(r"//.*", "", mv) and mv.count("__global__") == 1
    open(os.path.join(dst, "edge_general_kernel.cuh"), "w").write(mv)

    with open(os.path.join(CSRC, "sweep_phase.cuh")) as f:
        phase = f.read()
    assert "__shared__" not in phase and "asm" not in re.sub(r"//.*", "", phase)
    open(os.path.join(dst, "sweep_phase.cuh"), "w").write(phase)

    st = open(os.path.join(CSRC, "sweep_stencil.cu")).read()
    kernels = _cut(st, "template <int DIM, bool PMJ, int K, int ROUNDS, int V>\nstatic void sweep_launch_phase(", None,
                   "launchers of sweep_stencil.cu")
    i = st.find("static void stencil_block_shape(")
    k = st.find("template <int V>\nstatic int sweep_dispatch_kind(")
    assert 0 <= i < k
    shape = st[i:k]
    i = st.find("constexpr int NS_NP = 10;")
    k = st.find("template <int V>\nstatic int nsat_dispatch(")
    assert 0 <= i < k
    st = kernels + shape + st[i:k] + "\n}  // namespace ising\n"
    dyn = "    extern __shared__ uint32_t sm[];"
    assert st.count(dyn) == 4
    st = st.replace(dyn, "    uint32_t* sm = emu::dyn_smem;")
    assert st.count("__shared__") == 1            # the cooperative kernel's thresholds of the current sweep
    st = st.replace("__shared__", "EMU_SHARED")
    assert "asm" not in re.sub(r"//.*", "", st) and "<<<" not in st and st.count("__global__") == 4
    open(os.path.join(dst, "stencil_kernels.cuh"), "w").write(st)

    cl = open(os.path.join(CSRC, "sweep_cluster.cu")).read()
    cl = _cut(cl, "static_assert(sizeof(MscThresholds) / 4 <= 32", None, "launchers of sweep_cluster.cu") + \
        "\n}  // namespace ising\n"
    for ptx in ('    asm volatile("griddepcontrol.launch_dependents;");\n',
                '    asm volatile("griddepcontrol.wait;" ::: "memory");\n'):
        assert cl.count(ptx) == 1, ptx
        cl = cl.replace(ptx, "")
    assert cl.count(dyn) == 1
    cl = cl.replace(dyn, "    uint32_t* sm = emu::dyn_smem;")
    assert cl.count("__shared__") == 1            # th[2]: this sweep's and the next sweep's thresholds
    cl = cl.replace("__shared__", "EMU_SHARED")
    assert "asm" not in re.sub(r"//.*", "", cl) and cl.count("__global__") == 1
    open(os.path.join(dst, "cluster_kernel.cuh"), "w").write(cl)

    with open(os.path.join(CSRC, "pt_exp.h")) as f:
        open(os.path.join(dst, "pt_exp.h"), "w").write(f.read())
    pt = open(os.path.join(CSRC, "pt_device.cu")).read()
    pt, nwrap = re.subn(r"\nint launch_\w+\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", pt)
    assert nwrap == 4 and "<<<" not in pt and "launch_pdl" not in pt, nwrap
    for ptx in ('    asm volatile("griddepcontrol.launch_dependents;");\n',
                '    asm volatile("griddepcontrol.wait;" ::: "memory");\n'):
        assert pt.count(ptx) == 1, ptx
        pt = pt.replace(ptx, "")
    assert pt.count("__shared__") == 2            # the swap counters of k_pt_swap and k_pt_cycle (one block each)
    pt = pt.replace("__shared__", "EMU_SHARED")
    assert "asm" not in re.sub(r"//.*", "", pt)
    open(os.path.join(dst, "pt_device_kernels.cuh"), "w").write(pt)

    g2 = open(os.path.join(CSRC, "sweep_general.cu")).read()
    i = g2.find("// per-replica threshold tables from host-computed 64-bit thresholds")
    k = g2.find("// ------------------------------------------------------------------------------------------\n"
                "// Colour-class sweep for arbitrary real couplings and biases")
    assert 0 <= i < k
    g2, nwrap = re.subn(r"\nint launch_\w+\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", g2[i:k])
    assert nwrap == 3 and "<<<" not in g2 and g2.count("__global__") == 3, nwrap
    assert g2.count("__shared__") == 1            # the per-bit counters of k_nsat_general
    g2 = '#include "msc_device.cuh"\nnamespace ising {\n' + g2.replace("__shared__", "EMU_SHARED") + "\n}  // namespace ising\n"
    open(os.path.join(dst, "general_aux_kernels.cuh"), "w").write(g2)

    ob = open(os.path.join(CSRC, "observables.cu")).read()
    ob, nwrap = re.subn(r"\nint launch_\w+\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", ob)
    assert nwrap == 7 and "<<<" not in ob and ob.count("__global__") == 7, nwrap
    assert ob.count("__shared__") == 1
    open(os.path.join(dst, "observables_kernels.cuh"), "w").write(ob.replace("__shared__", "EMU_SHARED"))

    g3 = open(os.path.join(CSRC, "sweep_general.cu")).read()
    i = g3.find("template <int ROUNDS>\n__global__ void __launch_bounds__(256)\nk_sweep_real(")
    assert i >= 0
    g3, nwrap = re.subn(r"\nint launch_\w+\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", g3[i:])
    assert nwrap == 2 and "<<<" not in g3 and g3.count("__global__") == 2, nwrap
    open(os.path.join(dst, "real_kernels.cuh"), "w").write('#include "msc_device.cuh"\nnamespace ising {\n' + g3)

    mv2 = open(os.path.join(CSRC, "moves.cu")).read()
    i = mv2.find(head)
    k = mv2.find("// word m of the worm's random stream")
    assert 0 <= i < k
    mv2, nwrap = re.subn(r"\nint launch_\w+\([^{]*\{\n(?:    .*\n|\n)*?\}\n", "\n", mv2[:i] + mv2[k:])
    assert nwrap == 2 and "<<<" not in mv2 and mv2.count("__global__") == 2, nwrap
    open(os.path.join(dst, "float_moves_kernels.cuh"), "w").write(mv2)

    launch = open(os.path.join(CSRC, "sweep_rows_launch.cuh")).read()
    launch = _cut(launch, "template <int DIM, bool PMJ, int K, int ROUNDS, int V, bool ACC, bool MULTIROW, bool COUNT,",
                  None, "launchers of sweep_rows_launch.cuh") + "\n}  // namespace ising\n"
    assert "rows_shape" in launch and "rows_partition" in launch
    open(os.path.join(dst, "sweep_rows_launch_shape.cuh"), "w").write(launch)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    import shutil

    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    if shutil.which("g++") is None or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA toolkit headers (vector types) to build the host emulation")
    build = str(tmp_path_factory.mktemp("host_emulation"))
    prepare_sources(os.path.join(build, "prepared"))
    so = os.path.join(build, "libemu_rows.so")
    # EMU_SANITIZE=thread builds the emulation under ThreadSanitizer (tests/host_emulation/racecheck.py)
    san = ["-fsanitize=" + os.environ["EMU_SANITIZE"], "-g"] if os.environ.get("EMU_SANITIZE") else []
    flags = ["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-pthread", "-w", "-I", EMU, "-I", build,
             "-I", cuda_inc] + san
    units = ["emu_rows", "emu_general", "emu_strip", "emu_state", "emu_moves", "emu_stencil", "emu_pt", "emu_aux", "emu_float"]
    procs = [subprocess.Popen(flags + ["-c", os.path.join(EMU, u + ".cpp"), "-o", os.path.join(build, u + ".o")],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for u in units]
    for u, pr in zip(units, procs):
        _, err = pr.communicate()
        assert pr.returncode == 0, u + ":\n" + err[-4000:]
    res = subprocess.run(["g++", "-shared", "-pthread"] + san[:1] + ["-o", so] + [os.path.join(build, u + ".o") for u in units],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    lib = C.CDLL(so)
    lib.emu_rows_phase.restype = C.c_int
    lib.emu_rows_phase.argtypes = [C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                   C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32,
                                   C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_int]
    lib.emu_general_group.restype = C.c_int
    lib.emu_general_group.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                      C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_double,
                                      C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_uint]
    lib.emu_strip_init_random.argtypes = [C.c_void_p] + [C.c_uint32] * 5 + [C.c_uint64, C.c_uint]
    lib.emu_strip_observables.argtypes = [C.c_void_p] + [C.c_uint32] * 6 + [C.c_void_p, C.c_uint]
    lib.emu_strip_unpack.argtypes = [C.c_void_p] + [C.c_uint32] * 5 + [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint]
    lib.emu_strip_fused.restype = C.c_int
    lib.emu_strip_fused.argtypes = [C.c_void_p, C.c_void_p] + [C.c_uint32] * 6 + [C.c_uint64, C.c_uint32, C.c_double, C.c_double,
                                                                                 C.c_uint32, C.c_uint32, C.c_uint32]
    lib.emu_strip_phase.restype = C.c_int
    lib.emu_strip_phase.argtypes = [C.c_void_p] + [C.c_uint32] * 7 + [C.c_uint64, C.c_uint32, C.c_double, C.c_double,
                                                                      C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32]
    lib.emu_stencil.restype = C.c_int
    lib.emu_stencil.argtypes = [C.c_int, C.c_int] + [C.c_uint32] * 4 + [C.c_int, C.c_void_p, C.c_uint32, C.c_void_p,
                                C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32]
    lib.emu_pt_cycle.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_double, C.c_uint64, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_uint32, C.c_int,
                                 C.c_void_p, C.c_void_p]
    lib.emu_pt_swap.argtypes = [C.c_void_p] * 5 + [C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32]
    lib.emu_build_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint]
    lib.emu_nsat_general.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
    lib.emu_count_up.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_int, C.c_uint]
    lib.emu_overlap_from_counts.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint64]
    lib.emu_energy_from_hist.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_uint64, C.c_int,
                                         C.c_void_p, C.c_uint32]
    lib.emu_energy_from_nsat.argtypes = [C.c_void_p, C.c_uint64, C.c_double, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                         C.c_uint64]
    lib.emu_sweep_real.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 4 + [C.c_uint32, C.c_float, C.c_uint32,
                                                                                           C.c_uint64, C.c_uint32, C.c_int,
                                                                                           C.c_void_p, C.c_void_p]
    lib.emu_energy_real.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 5
    lib.emu_edge_moves.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 8 + [C.c_uint32, C.c_float, C.c_uint32,
                                                                                           C.c_uint64, C.c_uint32, C.c_uint32,
                                                                                           C.c_int]
    lib.emu_worm_moves.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32] + \
        [C.c_void_p] * 4 + [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_float, C.c_uint32, C.c_uint64, C.c_int]
    lib.emu_edge_group.restype = C.c_int
    lib.emu_edge_group.argtypes = [C.c_void_p, C.c_uint32] + [C.c_void_p] * 6 + [C.c_uint32] * 4 + [
        C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_uint]
    lib.emu_replay.restype = C.c_uint
    lib.emu_replay.argtypes = [C.c_uint64] * 3 + [C.c_void_p] * 8 + [C.c_double]
    lay = [C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32]
    lib.emu_init_random.argtypes = [C.c_void_p] + lay + [C.c_uint64, C.c_uint32, C.c_uint]
    lib.emu_pack_states.argtypes = [C.c_void_p] + lay + [C.c_void_p, C.c_uint64, C.c_uint]
    lib.emu_unpack_states.argtypes = [C.c_void_p] + lay + [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint]
    lib.emu_init_broadcast.argtypes = [C.c_void_p] + lay + [C.c_void_p, C.c_uint]
    lib.emu_export_natural.argtypes = [C.c_void_p] + lay + [C.c_void_p, C.c_uint]
    lib.emu_import_natural.argtypes = [C.c_void_p] + lay + [C.c_void_p, C.c_uint]
    return lib


# ---- the library's stencil layout, restated from csrc/kernels.h (Layout) and api_core.cu ------------
def torus(dims, rng, pmj, j0):
    """-> a, b, j of the periodic lattice, site = x + Lx (y + Ly z), bond d of site n: n -> n + e_d"""
    Lx, Ly, Lz = dims
    z, y, x = np.meshgrid(np.arange(Lz), np.arange(Ly), np.arange(Lx), indexing="ij")
    n = (x + Lx * (y + Ly * z)).ravel()
    fwd = [((x + 1) % Lx + Lx * (y + Ly * z)).ravel(), (x + Lx * ((y + 1) % Ly + Ly * z)).ravel()]
    if Lz > 1:
        fwd.append((x + Lx * (y + Ly * ((z + 1) % Lz))).ravel())
    a = np.concatenate([n] * len(fwd)).astype(np.uint64)
    b = np.concatenate(fwd).astype(np.uint64)
    j = np.full(len(a), j0)
    if pmj:
        j = j * rng.choice([-1.0, 1.0], size=len(a))
    return a, b, j


def layout_index(dims):
    """word row of natural site n in spins[2][rows][Lxh] (the replica words follow)"""
    Lx, Ly, Lz = dims
    n = np.arange(Lx * Ly * Lz)
    x, r = n % Lx, n // Lx
    y, z = r % Ly, r // Ly
    c = (x + y + z) & 1
    return (c * (Ly * Lz) + r) * (Lx // 2) + (x >> 1), c


def pack(states, dims, W):
    E, N = states.shape
    bits = np.zeros((N, W * 32), dtype=np.uint8)
    bits[:, :E] = states.T
    words = (bits.reshape(N, W, 32).astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(axis=2, dtype=np.uint32)
    idx, _ = layout_index(dims)
    out = np.zeros((N, W), dtype=np.uint32)
    out[idx] = words
    return out


def unpack(words, dims, E):
    idx, _ = layout_index(dims)
    w = words[idx]                                                    # natural order [N, W]
    bits = (w[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1
    return bits.reshape(len(idx), -1)[:, :E].T.astype(bool)


def bond_masks(dims, a, b, j):
    """[2][halfN][8] as upload_stencil_masks (api_core.cu) lays them out: k = 0 the x neighbour stored
    at the same half-index, 1 the other x neighbour, 2 y-1, 3 y+1, 4 z-1, 5 z+1; all-ones iff J > 0"""
    Lx, Ly, Lz = dims
    N = Lx * Ly * Lz
    ndir = 3 if Lz > 1 else 2
    anti = (j > 0).reshape(ndir, N)                                   # anti[d, n]: bond n -> n + e_d
    idx, c = layout_index(dims)
    n = np.arange(N)
    x, r = n % Lx, n // Lx
    y, z = r % Ly, r // Ly
    p = x & 1                                                         # = (y + z + c) & 1
    xm = ((x - 1) % Lx) + Lx * r
    ym = x + Lx * ((y - 1) % Ly + Ly * z)
    zm = x + Lx * (y + Ly * ((z - 1) % Lz))
    m = np.zeros((N, 8), dtype=np.uint32)
    jxp, jxm = anti[0, n], anti[0, xm]
    m[:, 0] = np.where(p == 0, jxp, jxm)
    m[:, 1] = np.where(p == 0, jxm, jxp)
    m[:, 2] = anti[1, ym]
    m[:, 3] = anti[1, n]
    if ndir == 3:
        m[:, 4] = anti[2, zm]
        m[:, 5] = anti[2, n]
    out = np.zeros((N, 8), dtype=np.uint32)
    out[idx] = m * np.uint32(0xFFFFFFFF)
    return out


def satisfied_bonds(states, a, b, j):
    s = states.astype(np.int64) * 2 - 1
    return ((s[:, a.astype(np.int64)] * s[:, b.astype(np.int64)] * np.sign(j)[None, :]) < 0).sum(axis=1)


CASES = [
    # dims, E, V, pmj, small, grid blocks, betas
    ((8, 6, 4), 128, 4, True, False, 5, [0.1, 0.5, 1.2]),      # config 3's instantiation (V = 4, +-J, 3D)
    ((8, 6, 4), 128, 4, True, True, 3, [0.3, 0.9]),            # ... in the 128-thread shape (the 8-GPU split)
    ((4, 4, 6), 96, 1, True, False, 7, [0.2, 0.7]),            # ragged last word (96 = 3 words), V = 1
    ((6, 4, 2), 64, 2, False, False, 2, [0.25, 0.6]),          # uniform ferromagnet, V = 2, Lz = 2 (z-1 == z+1)
    ((16, 8, 1), 128, 4, False, False, 4, [0.3, 0.44, 0.6]),   # config 2's instantiation (2D, uniform)
    ((12, 6, 1), 40, 2, True, False, 3, [0.4, 1.0]),           # 2D +-J, E not a multiple of 32
    ((600, 2, 1), 32, 1, False, False, 6, [0.44]),             # several x tiles per row, single row per unit
]


@pytest.mark.parametrize("dims,E,V,pmj,small,grid,betas", CASES)
def test_row_walk_source_equals_the_mirror(emu, oracle, dims, E, V, pmj, small, grid, betas):
    rng = np.random.default_rng(hash((dims, E, V, pmj)) & 0xFFFF)
    dim = 3 if dims[2] > 1 else 2
    j0 = -1.0 if pmj or dims[0] != 6 else 1.0                    # one uniform case is antiferromagnetic
    a, b, j = torus(dims, rng, pmj, j0)
    N = dims[0] * dims[1] * dims[2]
    _, colors = layout_index(dims)
    W = (E + 31) // 32
    if W % V:
        W += V - W % V                                            # the launcher picks V from W; pad words are idle replicas
    init = rng.integers(0, 2, size=(E, N)).astype(bool)
    seed, sweep0, gw0 = 0x1234567887654321, 5, 3
    words = pack(init, dims, W)
    jm8 = bond_masks(dims, a, b, j) if pmj else None
    antiferro = 0xFFFFFFFF if (not pmj and j0 > 0) else 0
    nsat_per_sweep = []
    for s, beta in enumerate(betas):
        for colour in (0, 1):
            nsat = np.zeros(W * 32, dtype=np.uint64)
            rc = emu.emu_rows_phase(dim, dims[0], dims[1], dims[2], W, V,
                                    None if jm8 is None else jm8.ctypes.data, antiferro, words.ctypes.data,
                                    colour, seed, sweep0 + s, gw0, float(beta), 1.0, int(colour == 1),
                                    nsat.ctypes.data, int(small), grid)
            assert rc == 0, rc
        nsat_per_sweep.append(nsat[:E].copy())
    got = unpack(words, dims, E)
    en_ref, st_ref = oracle.msc_mirror(a, b, j, N, colors, E, seed, betas, replica_offset=32 * gw0,
                                       states=init, sweep0=sweep0, per_sweep=True)
    assert (got == st_ref).all(), "kernel source on the host differs from the mirror"
    assert (got != init).mean() > 0.05                             # (the sweeps did move the spins)
    # the accumulating phase: satisfied bonds after every sweep <-> the mirror's per-sweep energies
    nb = len(a)
    en = np.array([(nb - 2.0 * n.astype(np.float64)) for n in nsat_per_sweep]).T
    assert (en == en_ref).all()
    assert (nsat_per_sweep[-1] == satisfied_bonds(got, a, b, j)).all()
    # and the count-only pass (get_energy of the current configuration)
    nsat = np.zeros(W * 32, dtype=np.uint64)
    rc = emu.emu_rows_phase(dim, dims[0], dims[1], dims[2], W, V, None if jm8 is None else jm8.ctypes.data,
                            antiferro, words.ctypes.data, 0, seed, 0, gw0, 0.0, 1.0, 2, nsat.ctypes.data, 0, grid)
    assert rc == 0, rc
    assert (nsat[:E] == satisfied_bonds(got, a, b, j)).all()
    assert (unpack(words, dims, E) == got).all()                  # count only: no update


# ---- general graphs (config 4's kernel) -----------------------------------------------------------------
def random_regular(n, d, rng):
    """pairing model, self-loops and double edges rejected (SURVEY 8(d), config 4)"""
    while True:
        stubs = rng.permutation(np.repeat(np.arange(n), d))
        a, b = stubs[0::2], stubs[1::2]
        if (a != b).all() and len({(min(x, y), max(x, y)) for x, y in zip(a, b)}) == len(a):
            return a.astype(np.uint64), b.astype(np.uint64)


def random_sparse(n, m, rng, max_deg):
    edges, deg = set(), np.zeros(n, dtype=int)
    while len(edges) < m:
        x, y = (int(v) for v in rng.integers(0, n, size=2))
        if x != y and (min(x, y), max(x, y)) not in edges and deg[x] < max_deg and deg[y] < max_deg:
            edges.add((min(x, y), max(x, y)))
            deg[x] += 1
            deg[y] += 1
    e = np.array(sorted(edges), dtype=np.uint64)
    return e[:, 0].copy(), e[:, 1].copy()


def greedy_colouring(n, a, b):
    adj = [[] for _ in range(n)]
    for x, y in zip(a.astype(int), b.astype(int)):
        adj[x].append(y)
        adj[y].append(x)
    col = np.full(n, -1)
    for v in range(n):
        used = {col[u] for u in adj[v]}
        col[v] = next(c for c in range(n) if c not in used)
    return col.astype(np.uint32), adj


def colour_degree_groups(n, a, b, j, col, adj):
    """(colour, degree) groups in the ELL form of kernels.h (GenGroup), colours ascending"""
    sign = {}
    for x, y, w in zip(a.astype(int), b.astype(int), j):
        sign[(x, y)] = sign[(y, x)] = w > 0
    groups = []
    for c in range(int(col.max()) + 1):
        for d in sorted({len(adj[v]) for v in range(n) if col[v] == c}):
            sites = np.array([v for v in range(n) if col[v] == c and len(adj[v]) == d], dtype=np.uint32)
            nbr = np.zeros((max(d, 1), len(sites)), dtype=np.uint32)
            anti = np.zeros(len(sites), dtype=np.uint32)
            for i, v in enumerate(sites):
                for k, u in enumerate(adj[v]):
                    nbr[k, i] = u
                    anti[i] |= np.uint32(int(sign[(int(v), u)]) << k)
            groups.append((d, sites, nbr, anti))
    return groups


def per_replica_tables(betas, W, K, jabs):
    """GenTables (kernels.h) from per-replica betas: what k_build_tables makes of the host's T64 rows"""
    import math

    plane = np.zeros((16, W, 8, 8), dtype=np.uint32)
    low = np.zeros((16, 32 * W, 8), dtype=np.uint32)
    for deg in range(16):
        cmin, ncls = deg // 2 + 1, deg - deg // 2
        for cls in range(min(ncls, 8)):
            de = 2.0 * jabs * (2 * (cmin + cls) - deg)
            for e, beta in enumerate(betas):
                scaled = math.ldexp(math.exp(-beta * de), K + 32)
                T = min(int(math.floor(scaled)), (1 << (K + 32)) - 1)
                low[deg, e, cls] = T & 0xFFFFFFFF
                for p in range(K):
                    plane[deg, e // 32, cls, p] |= np.uint32(((T >> (K + 31 - p)) & 1) << (e % 32))
    return plane, low


def pack_natural(states, W):
    E, N = states.shape
    bits = np.zeros((N, W * 32), dtype=np.uint8)
    bits[:, :E] = states.T
    return (bits.reshape(N, W, 32).astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(axis=2, dtype=np.uint32)


def unpack_natural(words, E):
    bits = (words[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1
    return bits.reshape(words.shape[0], -1)[:, :E].T.astype(bool)


GENERAL_CASES = [
    # graph, E, planes, rounds, per-replica betas, degree-specialised kernels, blocks
    ("3-regular", 64, 6, 7, True, True, 3),      # config 4: one beta per replica bit, V = 2, DEG = 3
    ("3-regular", 96, 6, 7, False, True, 64),    # uniform beta, V = 1
    ("3-regular", 64, 6, 7, False, False, 2),    # the run-time-degree kernel on the same graph
    ("mixed", 64, 6, 7, True, True, 5),          # degrees 1 .. 9: up to 5 uphill classes, +-J
    ("mixed", 32, 7, 10, False, False, 4),       # 7 planes, Philox4x32-10
    ("mixed", 64, 5, 7, False, False, 4),        # 5 planes (3 spare words for ties)
    ("cubic", 64, 6, 7, False, True, 7),         # a 4 x 4 x 4 torus as a general graph: DEG = 6
    ("square", 128, 6, 10, False, False, 3),     # DEG = 4 sites through the run-time-degree kernel, 10 rounds
]


@pytest.mark.parametrize("graph,E,K,rounds,perbeta,specialise,blocks", GENERAL_CASES)
def test_general_graph_source_equals_the_mirror(emu, oracle, graph, E, K, rounds, perbeta, specialise, blocks):
    rng = np.random.default_rng(len(graph) * 1000 + E + K)
    if graph == "3-regular":
        n = 200
        a, b = random_regular(n, 3, rng)
        j = np.full(len(a), -1.0)
    elif graph == "mixed":
        n = 120
        a, b = random_sparse(n, 300, rng, 9)
        j = rng.choice([-0.5, 0.5], size=len(a))
    elif graph == "cubic":
        a, b, j = torus((4, 4, 4), rng, True, -1.0)
        n = 64
    else:
        a, b, j = torus((6, 4, 1), rng, False, 2.0)
        n = 24
    jabs = float(abs(j[0]))
    col, adj = greedy_colouring(n, a, b)
    groups = colour_degree_groups(n, a, b, j, col, adj)
    W = (E + 31) // 32
    V = 2 if W % 2 == 0 else 1
    init = rng.integers(0, 2, size=(E, n)).astype(bool)
    words = pack_natural(init, W)
    seed, sweep0, gw0, nsweeps = 0xC0FFEE1234, 11, 2, 3
    if perbeta:
        betas_e = np.geomspace(0.1, 1.5, E)
        plane, low = per_replica_tables(betas_e, W, K, jabs)
        tp, tl = plane.ctypes.data, low.ctypes.data
        sweep_betas = [0.0] * nsweeps
    else:
        tp = tl = None
        sweep_betas = [0.2, 0.6, 1.1]
    for s, beta in enumerate(sweep_betas):
        for d, sites, nbr, anti in groups:
            rc = emu.emu_general_group(words.ctypes.data, W, V, sites.ctypes.data, nbr.ctypes.data, anti.ctypes.data,
                                       len(sites), d, sweep0 + s, seed, gw0, K, rounds, float(beta), jabs, tp, tl,
                                       int(specialise), blocks)
            assert rc == 0, rc
    got = unpack_natural(words, E)
    kw = dict(replica_offset=32 * gw0, planes=K, rounds=rounds, states=init, sweep0=sweep0)
    if perbeta:
        _, st_ref = oracle.msc_mirror(a, b, j, n, col, E, seed, None, per_replica_beta=betas_e, nsweeps=nsweeps, **kw)
    else:
        _, st_ref = oracle.msc_mirror(a, b, j, n, col, E, seed, sweep_betas, **kw)
    assert (got == st_ref).all(), "kernel source on the host differs from the mirror"
    assert (got != init).mean() > 0.05


# ---- one lattice bit-packed along x in row strips (config 5's kernel) ---------------------------------------
def strip_pack(state, Wr):
    """bool[rows, Lx] (global rows y0 ..) -> words[2][rows][Wr]: bit b of word j of colour c of global
    row y is site x = 2 (32 j + b) + ((y + c) & 1)  (kernels.h, StripGeom).  Needs y0 even."""
    rows, Lx = state.shape
    out = np.zeros((2, rows, Wr), dtype=np.uint32)
    for c in range(2):
        for r in range(rows):
            xs = 2 * np.arange(Lx // 2) + ((r + c) & 1)
            out[c, r] = (state[r, xs].reshape(Wr, 32).astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(
                axis=1, dtype=np.uint32)
    return out


def strip_unpack(words, Lx):
    _, rows, Wr = words.shape
    st = np.zeros((rows, Lx), dtype=bool)
    for c in range(2):
        for r in range(rows):
            xs = 2 * np.arange(Lx // 2) + ((r + c) & 1)
            st[r, xs] = ((words[c, r][:, None] >> np.arange(32, dtype=np.uint32)) & 1).ravel().astype(bool)
    return st


@pytest.mark.parametrize("Lx,Ly,nstrips,K,rounds,j", [(256, 12, 1, 6, 7, -1.0), (128, 16, 2, 6, 7, 1.0),
                                                      (192, 8, 2, 7, 10, -1.0), (64 * 40, 6, 1, 5, 7, -1.0)])
def test_strip_source_equals_the_mirror(emu, oracle, Lx, Ly, nstrips, K, rounds, j):
    rng = np.random.default_rng(Lx + Ly)
    Wr = Lx // 64
    init = rng.integers(0, 2, size=(Ly, Lx)).astype(bool)
    betas = [0.3, 0.44, 0.7]
    seed = 0xABCDEF0123456789
    full = strip_pack(init, Wr)                                   # [2][Ly][Wr]
    rows = Ly // nstrips                                          # even, so local parities are the global ones
    assert rows % 2 == 0
    strips = []
    for k in range(nstrips):
        buf = np.zeros((2, rows + 2, Wr), dtype=np.uint32)        # ghost = 1
        buf[:, 1:-1] = full[:, k * rows:(k + 1) * rows]
        strips.append(buf)

    def exchange(c):                                              # ghost rows of colour c from the neighbours
        for k, buf in enumerate(strips):
            buf[c, 0] = strips[(k - 1) % nstrips][c, rows]
            buf[c, rows + 1] = strips[(k + 1) % nstrips][c, 1]

    for t, beta in enumerate(betas):
        for c in (0, 1):
            exchange(1 - c)
            for k, buf in enumerate(strips):
                rc = emu.emu_strip_phase(buf.ctypes.data, Wr, rows, k * rows, Ly, 1, c, t, seed,
                                         0xFFFFFFFF if j > 0 else 0, float(beta), abs(j), K, rounds, 1, rows, 2 + k)
                assert rc == 0, rc
    got = strip_unpack(np.concatenate([b[:, 1:-1] for b in strips], axis=1), Lx)
    _, ref = oracle.msc_mirror_single(Lx, Ly, j, seed, betas, planes=K, rounds=rounds, state=init)
    assert (got == ref).all(), "kernel source on the host differs from the mirror"
    assert (got != init).mean() > 0.05


# ---- state initialisation / conversion and the replay kernel (csrc/state_io.cu) -----------------------------
@pytest.mark.parametrize("dims,E", [((8, 6, 4), 100), ((10, 4, 1), 33), (None, 70)])
def test_state_kernels_on_the_host(emu, oracle, dims, E):
    """k_init_random == the mirror's initial state; k_pack_states / k_unpack_states / k_init_broadcast
    against numpy, in the stencil layouts and in the natural-order layout of general graphs"""
    rng = np.random.default_rng(E)
    if dims is None:
        kind, n, lay3 = emu.emu_kind(0), 203, (0, 0, 0)           # general graph: natural order, odd nvars
        a = np.arange(n - 1, dtype=np.uint64)
        b = a + 1
        colors = (np.arange(n) & 1).astype(np.uint32)
    else:
        kind = emu.emu_kind(3 if dims[2] > 1 else 2)
        n, lay3 = dims[0] * dims[1] * dims[2], dims
        a, b, _ = torus(dims, rng, False, -1.0)
        _, colors = layout_index(dims)
    W = (E + 31) // 32
    seed, gw0 = 0x0123456789ABCDEF, 4
    lay = (kind, lay3[0], lay3[1], lay3[2], n, W)

    def unpack_k(words, stride=None):
        stride = n if stride is None else stride
        out = np.full((E, stride), 7, dtype=np.uint8)
        emu.emu_unpack_states(words.ctypes.data, *lay, out.ctypes.data, E, stride, 3)
        assert (out[:, n:] == 7).all()                            # nothing written beyond a row
        return out[:, :n].astype(bool)

    words = np.zeros(n * W, dtype=np.uint32)
    emu.emu_init_random(words.ctypes.data, *lay, seed, gw0, 2)
    _, st_ref = oracle.msc_mirror(a, b, np.full(len(a), -1.0), n, colors, E, seed, [], replica_offset=32 * gw0)
    assert (unpack_k(words) == st_ref).all()
    assert (unpack_k(words, stride=n + 5) == st_ref).all()        # the scalar store path (unaligned rows)

    states = rng.integers(0, 2, size=(E, n)).astype(np.uint8)
    words2 = np.zeros(n * W, dtype=np.uint32)
    emu.emu_pack_states(words2.ctypes.data, *lay, states.ctypes.data, E, 5)
    assert (unpack_k(words2) == states.astype(bool)).all()
    if dims is not None:
        assert (words2.reshape(n, W) == pack(states.astype(bool), dims, W)).all()      # Layout as documented
    else:
        assert (words2.reshape(n, W) == pack_natural(states.astype(bool), W)).all()
    nat = np.zeros((n, W), dtype=np.uint32)                       # packed words in natural site order and back
    emu.emu_export_natural(words2.ctypes.data, *lay, nat.ctypes.data, 2)
    assert (nat == pack_natural(states.astype(bool), W)).all()
    words3 = np.zeros(n * W, dtype=np.uint32)
    emu.emu_import_natural(words3.ctypes.data, *lay, nat.ctypes.data, 3)
    assert (words3 == words2).all()
    one = rng.integers(0, 2, size=n).astype(np.uint8)
    emu.emu_init_broadcast(words2.ctypes.data, *lay, one.ctypes.data, 1)
    assert (unpack_k(words2) == one.astype(bool)[None, :]).all()


def csr_sorted(n, a, b, j):
    """adjacency both ways, neighbours ascending, ties in edge-list order (graph.h: HostGraph)"""
    src = np.concatenate([a, b]).astype(np.int64)
    dst = np.concatenate([b, a]).astype(np.int64)
    w = np.concatenate([j, j])
    order = np.lexsort((np.concatenate([np.arange(len(a))] * 2), dst, src))
    row = np.zeros(n + 1, dtype=np.uint64)
    np.add.at(row, src + 1, 1)
    return np.cumsum(row).astype(np.uint64), dst[order].astype(np.uint32), w[order].copy()


@pytest.mark.parametrize("case", ["config1", "real"])
def test_replay_kernel_source_equals_the_reference_restatement(emu, oracle, case):
    """K1 on the host: the oracle (the reference algorithm restated, oracle/ising_oracle.c) emits its
    own (site, uniform) trace; the kernel source must land on the same states and energies."""
    rng = np.random.default_rng(3)
    if case == "config1":                                         # BASELINE config 1, shortened
        edges = oracle.square_edges(32)
        og = oracle.Graph(edges)
        beta, E, A = 0.44, 16, 30 * 1024
        bias = np.zeros(og.nvars)
    else:                                                         # real couplings and biases
        n = 40
        a0, b0 = random_sparse(n, 90, rng, 8)
        edges = [((int(x), int(y)), float(w)) for x, y, w in zip(a0, b0, rng.normal(size=len(a0)))]
        bias = rng.normal(size=n) * 0.3
        og = oracle.Graph(edges, biases=bias)
        beta, E, A = 0.8, 130, 4000
    n = og.nvars
    a = np.array([e[0][0] for e in edges], dtype=np.uint64)
    b = np.array([e[0][1] for e in edges], dtype=np.uint64)
    j = np.array([e[1] for e in edges], dtype=np.float64)
    seeds = rng.integers(0, 2**63, size=E).astype(np.uint64)
    sites, u, init, en_o, st_o = og.trace(beta, seeds, A)
    row, nbr, jv = csr_sorted(n, a, b, j)
    states = np.ascontiguousarray(init, dtype=np.uint8).copy()
    energies = np.zeros(E)
    bias = np.ascontiguousarray(bias, dtype=np.float64)
    amb = emu.emu_replay(E, n, A, row.ctypes.data, nbr.ctypes.data, jv.ctypes.data, bias.ctypes.data,
                         sites.ctypes.data, u.ctypes.data, states.ctypes.data, energies.ctypes.data, beta)
    assert amb == 0
    assert (states.astype(bool) == st_o).all()
    assert (energies == en_o).all()


# ---- bit-sliced two-spin edge moves (csrc/moves.cu: k_edge_general) -----------------------------------------
def strong_edge_colouring(n, a, b):
    """greedy: two bonds of a class share no site and no bond joins them (graph.h: EdgeClasses)"""
    adj = [set() for _ in range(n)]
    for x, y in zip(a.astype(int), b.astype(int)):
        adj[x].add(y)
        adj[y].add(x)
    cls = np.zeros(len(a), dtype=np.uint32)
    members = []                                                  # per class: set of sites blocked (ends + their neighbours)
    for e, (x, y) in enumerate(zip(a.astype(int), b.astype(int))):
        for c, blocked in enumerate(members):
            if x not in blocked and y not in blocked:
                break
        else:
            members.append(set())
            c = len(members) - 1
        cls[e] = c
        members[c] |= {x, y} | adj[x] | adj[y]
    return cls


def edge_groups(n, a, b, j, cls):
    """(class, outer degree) groups in the ELL form of kernels.h (EdgeGroup), natural-order slots"""
    inc = [[] for _ in range(n)]                                  # (far end, J > 0) per adjacency entry
    for x, y, w in zip(a.astype(int), b.astype(int), j):
        inc[x].append((y, w > 0))
        inc[y].append((x, w > 0))
    out = []
    for c in range(int(cls.max()) + 1):
        per_deg = {}
        for e in np.nonzero(cls == c)[0]:
            x, y = int(a[e]), int(b[e])
            outer = [(u, anti, 0) for u, anti in inc[x] if u != y] + [(u, anti, 1) for u, anti in inc[y] if u != x]
            per_deg.setdefault(len(outer), []).append((x, y, int(e), outer))
        for d in sorted(per_deg):
            items = per_deg[d]
            g = dict(sa=np.array([i[0] for i in items], dtype=np.uint32), sb=np.array([i[1] for i in items], dtype=np.uint32),
                     eid=np.array([i[2] for i in items], dtype=np.uint32), anti=np.zeros(len(items), dtype=np.uint32),
                     endp=np.zeros(len(items), dtype=np.uint32), nbr=np.zeros((max(d, 1), len(items)), dtype=np.uint32), deg=d)
            for i, (_, _, _, outer) in enumerate(items):
                for k, (u, anti, end) in enumerate(outer):
                    g["nbr"][k, i] = u
                    g["anti"][i] |= np.uint32(int(anti) << k)
                    g["endp"][i] |= np.uint32(end << k)
            out.append(g)
    return out


@pytest.mark.parametrize("graph,E,K,rounds,specialise", [("square", 64, 6, 7, True), ("3-regular", 96, 6, 7, True),
                                                         ("cubic", 64, 6, 7, True), ("mixed", 64, 6, 7, False),
                                                         ("mixed", 40, 5, 10, False), ("3-regular", 32, 7, 7, False)])
def test_edge_move_source_equals_the_mirror(emu, oracle, graph, E, K, rounds, specialise):
    rng = np.random.default_rng(E * K)
    if graph == "3-regular":
        n = 120
        a, b = random_regular(n, 3, rng)
        j = rng.choice([-1.0, 1.0], size=len(a))
    elif graph == "mixed":
        n = 80
        a, b = random_sparse(n, 130, rng, 6)
        j = rng.choice([-0.5, 0.5], size=len(a))
    elif graph == "cubic":
        a, b, j = torus((4, 4, 4), rng, True, -1.0)
        n = 64
    else:
        a, b, j = torus((8, 6, 1), rng, False, -1.0)
        n = 48
    jabs = float(abs(j[0]))
    cls = strong_edge_colouring(n, a, b)
    groups = edge_groups(n, a, b, j, cls)
    assert max(g["deg"] for g in groups) <= 15
    W = (E + 31) // 32
    init = rng.integers(0, 2, size=(E, n)).astype(bool)
    words = pack_natural(init, W)
    seed, gw0, betas, passes = 0x5EED5EED5EED, 1, [0.3, 0.8], 2
    for t, beta in enumerate(betas):
        for p in range(passes):
            for g in groups:
                rc = emu.emu_edge_group(words.ctypes.data, W, g["sa"].ctypes.data, g["sb"].ctypes.data,
                                        g["eid"].ctypes.data, g["anti"].ctypes.data, g["endp"].ctypes.data,
                                        g["nbr"].ctypes.data, len(g["sa"]), g["deg"], t, p, seed, gw0, K, rounds,
                                        float(beta), jabs, int(specialise), 3)
                assert rc == 0, rc
    got = unpack_natural(words, E)
    col, _ = greedy_colouring(n, a, b)
    _, ref = oracle.msc_mirror_moves(a, b, j, n, col, cls, E, seed, betas, spin_sweeps=0, edge_passes=passes,
                                     replica_offset=32 * gw0, planes=K, rounds=rounds, states=init)
    assert (got == ref).all(), "kernel source on the host differs from the mirror"
    assert (got != init).mean() > 0.05


# ---- the other checkerboard kernels: per-phase launch, cooperative chunk, cluster chunk, count only ---------
def stencil_tables(betas_e, W, dim, jabs, K=6):
    """per-replica tables of the lattice kernels: tplane[(w * 3 + cls) * 8 + p] bit b, tlow[(w * 32 + b) * 3 + cls]"""
    import math

    tplane = np.zeros((W, 3, 8), dtype=np.uint32)
    tlow = np.zeros((W * 32, 3), dtype=np.uint32)
    for e, beta in enumerate(betas_e):
        for c in range(dim):
            scaled = math.ldexp(math.exp(-beta * 4.0 * (c + 1) * jabs), K + 32)
            T = min(int(math.floor(scaled)), (1 << (K + 32)) - 1)
            tlow[e, c] = T & 0xFFFFFFFF
            for p in range(K):
                tplane[e // 32, c, p] |= np.uint32(((T >> (K + 31 - p)) & 1) << (e % 32))
    return tplane, tlow


STENCIL_CASES = [
    # mode, dims, E, V, pmj, K, rounds, per-replica betas, energies, SMs or CTAs of the cluster
    ("phase", (8, 6, 4), 128, 4, True, 5, 7, False, True, 2),
    ("phase", (8, 6, 4), 128, 4, True, 7, 10, False, False, 2),
    ("phase", (6, 4, 1), 20, 1, False, 7, 10, False, True, 3),
    ("phase", (4, 4, 4), 64, 2, False, 6, 7, True, True, 1),         # tempering on a lattice: one beta per replica bit
    ("phase", (12, 4, 1), 64, 2, True, 6, 7, True, False, 2),
    ("coop", (8, 4, 4), 128, 4, True, 6, 7, False, True, 5),
    ("coop", (16, 6, 1), 128, 4, False, 6, 7, False, False, 4),
    ("cluster", (8, 4, 4), 128, 4, True, 6, 7, False, True, 8),      # per-sweep energies (config 1's production path)
    ("cluster", (32, 32, 1), 32, 1, False, 6, 7, False, True, 16),   # BASELINE config 1's lattice, 16-CTA cluster
    ("cluster", (4, 4, 4), 32, 1, True, 6, 7, False, False, 8),
    ("cluster", (4, 4, 4), 64, 2, False, 6, 7, True, True, 8),       # tempering chunk ending with the counts
    ("cluster", (8, 6, 1), 64, 2, True, 6, 7, True, False, 4),
]


@pytest.mark.parametrize("mode,dims,E,V,pmj,K,rounds,perbeta,energies,units", STENCIL_CASES)
def test_checkerboard_kernels_equal_the_mirror(emu, oracle, mode, dims, E, V, pmj, K, rounds, perbeta, energies, units):
    rng = np.random.default_rng(sum(dims) * 7 + E + K)
    dim = 3 if dims[2] > 1 else 2
    a, b, j = torus(dims, rng, pmj, -1.0)
    N = dims[0] * dims[1] * dims[2]
    _, colors = layout_index(dims)
    W = (E + 31) // 32
    assert W % V == 0
    init = rng.integers(0, 2, size=(E, N)).astype(bool)
    words = pack(init, dims, W)
    jmask = None
    if pmj:                                                       # [2][2 dim][halfN]: the k-major form of the masks
        jmask = np.ascontiguousarray(bond_masks(dims, a, b, j).reshape(2, N // 2, 8)[:, :, :2 * dim].transpose(0, 2, 1))
    seed, sweep0, gw0, cw = 0xFEEDFACE12345, 9, 2, W * 32
    nsw = 3
    if perbeta:
        betas_e = np.geomspace(0.1, 1.4, E)
        tplane, tlow = stencil_tables(betas_e, W, dim, 1.0)
        tp, tl = tplane.ctypes.data, tlow.ctypes.data
        betas = np.zeros(nsw)
    else:
        tp = tl = None
        betas = np.array([0.2, 0.5, 1.0])
    jm = None if jmask is None else jmask.ctypes.data
    nb = len(a)

    def call(m, colour, sweep, n, bts, acc, hist):
        return emu.emu_stencil(m, dim, dims[0], dims[1], dims[2], W, V, jm, 0, words.ctypes.data, colour, seed, sweep, n,
                               gw0, K, rounds, bts.ctypes.data, 1.0, tp, tl, int(acc), hist.ctypes.data, cw, units)

    if mode == "phase":
        hist = np.zeros((nsw, cw), dtype=np.uint64)
        for t in range(nsw):
            for colour in (0, 1):
                assert call(0, colour, sweep0 + t, 1, betas[t:t + 1], energies and colour == 1, hist[t]) == 0
    else:
        last_only = perbeta                                       # a tempering chunk leaves the last sweep's counts
        hist = np.zeros((1 if last_only else nsw, cw), dtype=np.uint64)
        assert call(1 if mode == "coop" else 2, 0, sweep0, nsw, betas, energies, hist) == 0
    got = unpack(words, dims, E)
    kw = dict(replica_offset=32 * gw0, planes=K, rounds=rounds, states=init, sweep0=sweep0, per_sweep=True)
    if perbeta:
        en_ref, st_ref = oracle.msc_mirror(a, b, j, N, colors, E, seed, None, per_replica_beta=betas_e, nsweeps=nsw, **kw)
    else:
        en_ref, st_ref = oracle.msc_mirror(a, b, j, N, colors, E, seed, betas, **kw)
    assert (got == st_ref).all(), "kernel source on the host differs from the mirror"
    assert (got != init).mean() > 0.05
    if energies:
        en = nb - 2.0 * hist[:, :E].astype(np.float64).T
        if mode != "phase" and perbeta:
            assert (en[:, 0] == en_ref[:, -1]).all()
        else:
            assert (en == en_ref).all()
    # the count-only pass on the final configuration
    cnt = np.zeros(cw, dtype=np.uint64)
    assert call(3, 0, 0, 0, betas, 0, cnt) == 0
    assert (cnt[:E] == satisfied_bonds(got, a, b, j)).all()


# ---- a whole tempering run: cluster chunks + k_pt_cycle, as ising_pt_timesteps_sample enqueues them ----------
@pytest.mark.parametrize("dims,R,timesteps,swap_freq,sampling_freq,pmj", [((4, 4, 4), 32, 24, 3, 4, True),
                                                                          ((8, 4, 1), 20, 30, 5, 2, False),
                                                                          ((4, 4, 2), 64, 12, 1, 3, False)])
def test_tempering_run_on_the_host_equals_the_mirror(emu, oracle, native, dims, R, timesteps, swap_freq, sampling_freq, pmj):
    import math

    rng = np.random.default_rng(R + timesteps)
    dim = 3 if dims[2] > 1 else 2
    a, b, j = torus(dims, rng, pmj, -1.0)
    N, nb = dims[0] * dims[1] * dims[2], len(a)
    _, colors = layout_index(dims)
    W = (R + 31) // 32
    V = 2 if W % 2 == 0 else 1
    e32, K, seed = W * 32, 6, 0x7E57AB1E5EED
    betas = np.geomspace(0.15, 1.3, R)
    kind = emu.emu_kind(dim)
    words = np.zeros(N * W, dtype=np.uint32)
    emu.emu_init_random(words.ctypes.data, kind, dims[0], dims[1], dims[2], N, W, seed, 0, 2)
    jmask = None
    if pmj:
        jmask = np.ascontiguousarray(bond_masks(dims, a, b, j).reshape(2, N // 2, 8)[:, :, :2 * dim].transpose(0, 2, 1))
    # device-resident state of the ladder (api_pt.cu: ising_pt)
    slot_of_cfg = np.arange(R, dtype=np.uint32)
    cfg_of_slot = np.arange(R, dtype=np.uint32)
    gidx = np.arange(R, dtype=np.uint32)
    stats = np.zeros(2 + 2 * R, dtype=np.uint64)
    slot_of_replica = np.zeros(e32, dtype=np.uint32)
    slot_of_replica[:R] = np.arange(R)
    t64 = np.zeros((R, 3), dtype=np.uint64)                       # thresholds by SLOT (host-computed, libm exp)
    for s_, beta in enumerate(betas):
        for c in range(dim):
            t64[s_, c] = min(int(math.floor(math.ldexp(math.exp(-beta * 4.0 * (c + 1)), K + 32))), (1 << (K + 32)) - 1)
    tplane, tlow = stencil_tables(betas[slot_of_replica[:R]], W, dim, 1.0)
    nsat = np.zeros(e32, dtype=np.uint64)
    e_local, e_all, acc = np.zeros(e32), np.zeros(e32), np.zeros(R)
    ns = timesteps // sampling_freq
    samples = np.zeros((R, ns, N), dtype=bool)
    none = np.zeros(timesteps)                                    # (betas of a chunk: unused with per-replica tables)
    remaining, to_swap, to_sample, k, sweep = timesteps, swap_freq, sampling_freq, 0, 0
    while remaining > 0:                                          # ising_pt_timesteps_sample's loop
        t = min(to_sample, to_swap, remaining)
        rc = emu.emu_stencil(2, dim, dims[0], dims[1], dims[2], W, V, None if jmask is None else jmask.ctypes.data, 0,
                             words.ctypes.data, 0, seed, sweep, t, 0, K, 7, none.ctypes.data, 1.0, tplane.ctypes.data,
                             tlow.ctypes.data, 1, nsat.ctypes.data, e32, 8)
        assert rc == 0, rc
        sweep += t
        to_sample -= t
        to_swap -= t
        remaining -= t
        emu.emu_pt_cycle(nsat.ctypes.data, e_local.ctypes.data, e_all.ctypes.data, R, e32, 1.0, nb, 2, gidx.ctypes.data,
                         betas.ctypes.data, slot_of_cfg.ctypes.data, cfg_of_slot.ctypes.data, R, seed, stats.ctypes.data,
                         slot_of_replica.ctypes.data, acc.ctypes.data, float(t), int(to_swap == 0),
                         t64.ctypes.data if to_swap == 0 else None, W, K, tplane.ctypes.data, tlow.ctypes.data)
        assert (nsat == 0).all()                                  # zeroed for the next cycle
        if to_swap == 0:
            to_swap = swap_freq
        if to_sample == 0:
            if k < ns:
                samples[:, k, :] = unpack(words.reshape(N, W), dims, R)[cfg_of_slot]
            k += 1
            to_sample = sampling_freq
    st_ref, en_ref, swaps_ref, slots_ref = oracle.msc_mirror_pt(a, b, j, N, colors, betas, seed, timesteps, swap_freq,
                                                                sampling_freq)
    assert (samples == st_ref).all()
    assert (acc / timesteps == en_ref).all()
    assert int(stats[1]) == swaps_ref and int(stats[0]) == timesteps // swap_freq
    assert (slot_of_cfg == slots_ref).all()
    assert swaps_ref > 0
    # per-pair counters: every pair attempted once per swap step
    assert (stats[2:2 + R - 1] == timesteps // swap_freq).all() and int(stats[2 + R:].sum()) == swaps_ref

    # k_pt_swap alone == the host's ising_pt_decide_swaps on the same energies
    en = rng.normal(size=R) * 20
    s1, c1 = np.arange(R, dtype=np.uint32), np.arange(R, dtype=np.uint32)
    st1 = np.zeros(2 + 2 * R, dtype=np.uint64)
    st1[0] = 5
    emu.emu_pt_swap(betas.ctypes.data, en.ctypes.data, gidx.ctypes.data, s1.ctypes.data, c1.ctypes.data, R, seed,
                    st1.ctypes.data, slot_of_replica.ctypes.data, e32)
    s2, c2 = np.arange(R, dtype=np.uint32), np.arange(R, dtype=np.uint32)
    nsw = C.c_uint64(0)
    lib = native.lib()
    rc = lib.ising_pt_decide_swaps(betas.ctypes.data_as(C.c_void_p), C.c_uint64(R), en.ctypes.data_as(C.c_void_p),
                                   C.c_uint64(seed), C.c_uint64(5), s2.ctypes.data_as(C.c_void_p),
                                   c2.ctypes.data_as(C.c_void_p), C.byref(nsw))
    assert rc == 0
    assert (s1 == s2).all() and (c1 == c2).all() and int(st1[1]) == nsw.value and int(st1[0]) == 6


# ---- the smaller kernels around the sweeps ------------------------------------------------------------------
def test_table_builders_on_the_host(emu):
    """k_build_tables / k_build_tables_stencil (warp votes) == the tables the tests above build in numpy,
    under a non-trivial replica -> slot permutation"""
    import math

    rng = np.random.default_rng(11)
    R, W, K = 50, 2, 6
    betas = np.geomspace(0.1, 1.5, R)                              # by slot
    slot_of_replica = np.zeros(W * 32, dtype=np.uint32)
    slot_of_replica[:R] = rng.permutation(R)

    def t64_of(beta, de):
        return min(int(math.floor(math.ldexp(math.exp(-beta * de), K + 32))), (1 << (K + 32)) - 1)

    jabs = 0.5
    t64 = np.zeros((R, 16, 8), dtype=np.uint64)                    # general: [slot][deg][cls]
    for s_, beta in enumerate(betas):
        for deg in range(16):
            for cls in range(min(deg - deg // 2, 8)):
                t64[s_, deg, cls] = t64_of(beta, 2.0 * jabs * (2 * (deg // 2 + 1 + cls) - deg))
    plane = np.zeros((16, W, 8, 8), dtype=np.uint32)
    low = np.zeros((16, 32 * W, 8), dtype=np.uint32)
    emu.emu_build_tables(t64.ctypes.data, slot_of_replica.ctypes.data, W, K, plane.ctypes.data, low.ctypes.data, 0, 7)
    per_replica = np.concatenate([betas[slot_of_replica[:R]], np.full(W * 32 - R, betas[0])])   # padding bits: slot 0
    plane_ref, low_ref = per_replica_tables(per_replica, W, K, jabs)
    assert (plane == plane_ref).all() and (low == low_ref).all()

    t64s = np.zeros((R, 3), dtype=np.uint64)                       # lattices: [slot][cls]
    for s_, beta in enumerate(betas):
        for c in range(3):
            t64s[s_, c] = t64_of(beta, 4.0 * (c + 1) * jabs)
    tplane = np.zeros((W, 3, 8), dtype=np.uint32)
    tlow = np.zeros((W * 32, 3), dtype=np.uint32)
    emu.emu_build_tables(t64s.ctypes.data, slot_of_replica.ctypes.data, W, K, tplane.ctypes.data, tlow.ctypes.data, 1, 2)
    tp_ref, tl_ref = stencil_tables(per_replica, W, 3, jabs)
    assert (tplane == tp_ref).all() and (tlow == tl_ref).all()


@pytest.mark.parametrize("E", [37, 128])
def test_count_and_energy_kernels_on_the_host(emu, E):
    """get_energy on a general graph (k_nsat_general), magnetisation and pair overlaps (k_count_up),
    bond counts -> energies, against numpy"""
    rng = np.random.default_rng(E)
    n = 150
    a, b = random_sparse(n, 400, rng, 15)
    j = rng.choice([-1.5, 1.5], size=len(a))
    W = (E + 31) // 32
    states = rng.integers(0, 2, size=(E, n)).astype(bool)
    words = pack_natural(states, W)
    row, nbr, jv = csr_sorted(n, a, b, j)
    row32, anti = row.astype(np.uint32), (jv > 0).astype(np.uint8)
    nsat2 = np.zeros(W * 32, dtype=np.uint64)
    emu.emu_nsat_general(words.ctypes.data, n, W, row32.ctypes.data, nbr.ctypes.data, anti.ctypes.data, nsat2.ctypes.data, 3)
    sat = satisfied_bonds(states, a, b, j)
    assert (nsat2[:E] == 2 * sat).all()                           # every bond seen from both ends
    en = np.zeros((E, 3))
    emu.emu_energy_from_nsat(nsat2.ctypes.data, E, 1.5, len(a), 1, en.ctypes.data, 3, 1)
    s = states.astype(np.int64) * 2 - 1
    e_ref = (s[:, a.astype(int)] * s[:, b.astype(int)] * j[None, :]).sum(axis=1)
    assert (en[:, 1] == e_ref).all() and (en[:, 0] == 0).all() and (en[:, 2] == 0).all()

    up = np.zeros(W * 32, dtype=np.uint64)
    emu.emu_count_up(words.ctypes.data, n, W, up.ctypes.data, 0, 4)
    assert (up[:E] == states.sum(axis=1)).all()
    dis = np.zeros(W * 32, dtype=np.uint64)
    emu.emu_count_up(words.ctypes.data, n, W, dis.ctypes.data, 1, 4)
    P = E // 2
    q = np.zeros((P, 2))
    emu.emu_overlap_from_counts(dis.ctypes.data, P, n, q.ctypes.data, 2, 0)
    assert (q[:, 0] == (s[0:2 * P:2] * s[1:2 * P:2]).sum(axis=1)).all()

    nt, cw, copies = 4, W * 32, 3                                 # per-sweep histories spread over counter copies
    hist = rng.integers(0, 50, size=(nt, copies, cw)).astype(np.uint64)
    out = np.zeros((E, nt))
    emu.emu_energy_from_hist(hist.ctypes.data, E, cw, nt, 1.5, len(a), 2, out.ctypes.data, copies)
    assert (out == 1.5 * (len(a) - 2.0 * hist.sum(axis=1)[:, :E].T.astype(np.float64))).all()


# ---- the float-field kernels: statistics against exact enumeration ------------------------------------------
@pytest.mark.parametrize("moves", [False, True])
def test_float_kernels_on_the_host_sample_the_boltzmann_law(emu, moves):
    """k_sweep_real (real couplings, biases) alone, and with passes of float edge moves (importance
    weights included) and 4-site worm moves in every timestep: <E> and <m> within 4 sigma of the exact
    enumeration of the 2^10 states; k_energy_real against numpy."""
    rng = np.random.default_rng(17 + moves)
    n, E, beta = 10, 1024, 0.6
    a, b = random_sparse(n, 18, rng, 6)
    j = rng.normal(size=len(a))
    bias = rng.normal(size=n) * 0.4
    W = E // 32
    row, nbr, jv = csr_sorted(n, a, b, j)
    row32, jf, biasf = row.astype(np.uint32), jv.astype(np.float32), bias.astype(np.float32)
    col, _ = greedy_colouring(n, a, b)
    colour_sites = [np.nonzero(col == c)[0].astype(np.uint32) for c in range(int(col.max()) + 1)]
    cls = strong_edge_colouring(n, a, b)
    classes = []
    for c in range(int(cls.max()) + 1):
        ids = np.nonzero(cls == c)[0].astype(np.uint32)
        wrel = (np.abs(j[ids]) / np.abs(j).max()).astype(np.float32)
        classes.append((a[ids].astype(np.uint32), b[ids].astype(np.uint32), ids, wrel))
    # exact: E(s) = sum J s s - sum b s over all 2^n states, in the f32 couplings the kernels see
    st = ((np.arange(2 ** n)[:, None] >> np.arange(n)) & 1) * 2 - 1
    jq, bq = j.astype(np.float32).astype(np.float64), bias.astype(np.float32).astype(np.float64)
    en_all = (st[:, a.astype(int)] * st[:, b.astype(int)] * jq).sum(axis=1) - (st * bq).sum(axis=1)
    wgt = np.exp(-beta * (en_all - en_all.min()))
    wgt /= wgt.sum()
    e_exact, m_exact = (wgt * en_all).sum(), (wgt * st.sum(axis=1)).sum()

    words = pack_natural(rng.integers(0, 2, size=(E, n)).astype(bool), W)
    seed, burn, total, every = 0xF10A7, 22, 66, 4
    e_samples, m_samples = [], []
    for t in range(total):
        for sites in colour_sites:
            emu.emu_sweep_real(words.ctypes.data, sites.ctypes.data, len(sites), row32.ctypes.data, nbr.ctypes.data,
                               jf.ctypes.data, biasf.ctypes.data, W, beta, t, seed, 0, 7, None, None)
        if moves:
            for ea, eb, ids, wrel in classes:
                emu.emu_edge_moves(words.ctypes.data, n, W, row32.ctypes.data, nbr.ctypes.data, jf.ctypes.data,
                                   biasf.ctypes.data, ea.ctypes.data, eb.ctypes.data, ids.ctypes.data, wrel.ctypes.data,
                                   len(ids), beta, t, seed, 0, 0, 7)
            emu.emu_worm_moves(words.ctypes.data, 0, 0, 0, 0, n, W, row32.ctypes.data, nbr.ctypes.data, jf.ctypes.data,
                               biasf.ctypes.data, E, 0, 2, 4, beta, t, seed, 7)
        if t >= burn and (t - burn) % every == 0:
            en = np.zeros(W * 32)
            emu.emu_energy_real(words.ctypes.data, n, W, row32.ctypes.data, nbr.ctypes.data, jv.ctypes.data,
                                bias.ctypes.data, en.ctypes.data)
            s = unpack_natural(words, E).astype(np.int64) * 2 - 1
            ref = (s[:, a.astype(int)] * s[:, b.astype(int)] * j).sum(axis=1) - (s * bias).sum(axis=1)
            assert np.allclose(en, ref, rtol=0, atol=1e-10)
            e_samples.append(en)
            m_samples.append(s.sum(axis=1))
    for samples, exact in ((e_samples, e_exact), (m_samples, m_exact)):
        per_exp = np.mean(samples, axis=0)                        # experiments are independent chains
        err = per_exp.std(ddof=1) / np.sqrt(E)
        assert abs(per_exp.mean() - exact) < 4 * err + 2e-3, (per_exp.mean(), exact, err)


def float_test_graph(rng, n=240):
    """Gaussian couplings and biases over magnitudes 1e-3 .. 1e3, a hub of degree 120, a leaf, an
    isolated site (n - 1) and a double bond: what the statistical graphs above do not reach"""
    a, b = random_sparse(n - 2, 420, rng, 12)
    hub = np.arange(1, 121, dtype=np.uint64)
    a = np.concatenate([a, np.zeros(120, dtype=np.uint64), [n - 2, 5]]).astype(np.uint64)   # leaf n - 2; 0-5 twice
    b = np.concatenate([b, hub, [7, 0]]).astype(np.uint64)
    scale = np.where(rng.random(len(a)) < 0.3, 10.0 ** rng.uniform(-3, 3, len(a)), 1.0)
    j = rng.normal(size=len(a)) * scale
    bias = rng.normal(size=n) * 0.5 * np.where(rng.random(n) < 0.2, 10.0 ** rng.uniform(-3, 2, n), 1.0)
    bias[n - 1] = 0.0
    return a, b, j, bias


@pytest.mark.parametrize("E,rounds,gw0,perbeta", [(1, 7, 0, False), (5, 10, 2, False), (33, 7, 2, True),
                                                  (1031, 10, 0, True)])
def test_float_kernels_on_the_host_take_the_reference_decisions(emu, E, rounds, gw0, perbeta):
    """k_sweep_real, k_edge_moves and k_worm_moves from their source, launch by launch, against the f64
    reference of tests/float_reference.py: every decision outside the rounding band equals the reference's
    (bit for bit on every replica that met no in-band decision), and the band holds < 1e-3 of them.
    Philox rounds, the global word of local word 0, the worms' replica offset, per-replica betas through a
    permuted slot map that spans two words, W = 1 and W = 33 (two word columns per block)."""
    import float_reference as fr

    rng = np.random.default_rng(1000 + E)
    n = 240
    a, b, j, bias = float_test_graph(rng, n)
    W = (E + 31) // 32
    row, nbr, jv = csr_sorted(n, a, b, j)
    row32, jf, biasf = row.astype(np.uint32), jv.astype(np.float32), bias.astype(np.float32)
    col, _ = greedy_colouring(n, a, b)
    cls = strong_edge_colouring(n, a, b)
    g = fr.Graph(n, a, b, j, bias, col, cls)
    classes = [np.nonzero(col == c)[0].astype(np.uint32) for c in range(int(col.max()) + 1)]
    eclasses = []
    for c in range(int(cls.max()) + 1):
        ids = np.nonzero(cls == c)[0].astype(np.uint32)
        eclasses.append((a[ids].astype(np.uint32), b[ids].astype(np.uint32), ids, g.wrel[ids].astype(np.float32)))
    seed = 0x5EED0F10A7 + E
    init = rng.integers(0, 2, size=(E, n)).astype(bool)
    words = pack_natural(init, W)
    ch = fr.Chain(g, init, seed, rep0=32 * gw0, rounds=rounds)
    slots = slot_bits = None
    if perbeta:                                                   # slot map over all 32 W bits, permuted
        by_slot = rng.permutation(np.concatenate([[0.0, 1e6], np.linspace(0.05, 3.0, 32 * W - 2)]))
        slot_of_rep = rng.permutation(32 * W).astype(np.uint32)
        slot_bits = np.ascontiguousarray(by_slot).view(np.uint64)
        slots = slot_of_rep
        beta_rep = by_slot[slot_of_rep[:E]]
        assert W == 1 or len({float(x) for x in beta_rep[32:]} - {float(x) for x in by_slot[slot_of_rep[:E - 32]]}) > 0

    def check(what):
        got = unpack_natural(words, E)
        bad = np.nonzero((got != ch.s).any(axis=1) & ch.determined)[0]
        assert len(bad) == 0, f"{what}: replicas {bad[:10]} differ from the reference outside the band"

    for t, beta in enumerate([0.0, 0.3, 1.0, 3.0, 1e6]):
        for sites in classes:
            emu.emu_sweep_real(words.ctypes.data, sites.ctypes.data, len(sites), row32.ctypes.data, nbr.ctypes.data,
                               jf.ctypes.data, biasf.ctypes.data, W, beta, t, seed, gw0, rounds,
                               None if slots is None else slot_bits.ctypes.data,
                               None if slots is None else slots.ctypes.data)
        ch.sweep(t, beta_rep if perbeta else beta)
        check(f"sweep t={t}")
        for p in range(2):
            for ea, eb, ids, wrel in eclasses:
                emu.emu_edge_moves(words.ctypes.data, n, W, row32.ctypes.data, nbr.ctypes.data, jf.ctypes.data,
                                   biasf.ctypes.data, ea.ctypes.data, eb.ctypes.data, ids.ctypes.data,
                                   wrel.ctypes.data if p == 1 else None, len(ids), beta, t, seed, gw0, p, rounds)
            ch.edge_pass(t, beta, p, importance=p == 1)
            check(f"edge pass {p} t={t}")
        length = [1, 2, 5, 8, 3][t]
        emu.emu_worm_moves(words.ctypes.data, 0, 0, 0, 0, n, W, row32.ctypes.data, nbr.ctypes.data, jf.ctypes.data,
                           biasf.ctypes.data, E, 32 * gw0, 3, length, beta, t, seed, rounds)
        ch.worms(t, beta, 3, length)
        check(f"worms of {length} t={t}")
    assert ch.decisions > 0 and ch.in_band < 1e-3 * ch.decisions, (ch.in_band, ch.decisions)
    assert ch.determined.mean() > 0.9
    assert (unpack_natural(words, E) != init).any()


def test_worms_on_the_checkerboard_layout_take_the_reference_decisions(emu):
    """k_worm_moves addressing spins through the checkerboard layout of a torus (site_word_base), at a
    replica offset of 64, real couplings and a bias: the reference's decisions, bit for bit"""
    import float_reference as fr

    rng = np.random.default_rng(29)
    dims, E, offset, seed = (6, 4, 4), 70, 64, 0xC0FFEE
    a, b, _ = torus(dims, rng, False, 1.0)
    j = rng.normal(size=len(a))
    n = dims[0] * dims[1] * dims[2]
    bias = rng.normal(size=n) * 0.3
    W = (E + 31) // 32
    row, nbr, jv = csr_sorted(n, a, b, j)
    row32, jf, biasf = row.astype(np.uint32), jv.astype(np.float32), bias.astype(np.float32)
    g = fr.Graph(n, a, b, j, bias)
    init = rng.integers(0, 2, size=(E, n)).astype(bool)
    words = pack(init, dims, W)
    ch = fr.Chain(g, init, seed, rep0=offset, rounds=7)
    for t, (beta, length) in enumerate([(0.4, 3), (1.5, 5), (0.0, 2), (1e6, 4)]):
        emu.emu_worm_moves(words.ctypes.data, 3, dims[0], dims[1], dims[2], n, W, row32.ctypes.data, nbr.ctypes.data,
                           jf.ctypes.data, biasf.ctypes.data, E, offset, 4, length, beta, t, seed, 7)
        ch.worms(t, beta, 4, length)
        got = unpack(words, dims, E)
        assert not ((got != ch.s).any(axis=1) & ch.determined).any(), t
    assert ch.determined.all() and ch.in_band == 0
    assert (unpack(words, dims, E) != init).any()


def test_strip_state_kernels_on_the_host(emu, oracle):
    """k_strip_init_random == the mirror's Philox initial state (two strips of one lattice);
    k_strip_unpack and k_strip_observables against numpy"""
    Lx, Ly, seed, j = 192, 12, 0x51DE5EED, 1.0
    Wr, rows = Lx // 64, Ly // 2
    _, ref = oracle.msc_mirror_single(Lx, Ly, j, seed, [])        # no sweeps: the initial state
    full = strip_pack(ref, Wr)
    for k in range(2):
        buf = np.zeros((2, rows + 2, Wr), dtype=np.uint32)
        emu.emu_strip_init_random(buf.ctypes.data, Wr, rows, k * rows, Ly, 1, seed, 3)
        assert (buf[:, 1:-1] == full[:, k * rows:(k + 1) * rows]).all()
        assert (buf[:, 0] == 0).all() and (buf[:, -1] == 0).all()  # ghost rows come from the neighbours
        for c in range(2):
            buf[c, 0] = full[c, (k * rows - 1) % Ly]
            buf[c, -1] = full[c, ((k + 1) * rows) % Ly]
        out = np.zeros((rows - 1, Lx), dtype=np.uint8)
        emu.emu_strip_unpack(buf.ctypes.data, Wr, rows, k * rows, Ly, 1, out.ctypes.data, 1, rows - 1, 2)
        assert (out.astype(bool) == ref[k * rows + 1:(k + 1) * rows]).all()
        acc = np.zeros(2, dtype=np.uint64)
        emu.emu_strip_observables(buf.ctypes.data, Wr, rows, k * rows, Ly, 1, 0xFFFFFFFF, acc.ctypes.data, 2)
        # satisfied (antiferromagnetic: unequal) bonds seen from the colour-0 sites of the strip's rows; all up spins
        y = np.arange(k * rows, (k + 1) * rows)
        sat = 0
        for yy in y:
            xs = np.arange(Lx)[(np.arange(Lx) + yy) % 2 == 0]
            for dx, dy in ((1, 0), (-1, 0), (0, 1), (0, -1)):
                sat += int((ref[yy, xs] != ref[(yy + dy) % Ly, (xs + dx) % Lx]).sum())
        assert int(acc[0]) == sat and int(acc[1]) == int(ref[y].sum())


# ---- ledger: every kernel of the library is either run here from its source or named with the reason why not ----
NOT_EMULATED = {
    "k_sweep_rows_tma": "opt-in (ISING_TMA=1) variant staged by cp.async.bulk + mbarrier PTX; bit-identical to k_sweep_rows on the GPU",
    "k_strip_sweep_fused_tma": "opt-in (ISING_STRIP_FUSE=1), cp.async.bulk + mbarrier PTX",
    "k_pt_gather_rows": "row copy by index (slot-ordered samples); the tempering test above does the same gather in numpy",
    "k_pt_local_slots": "three-line index map, the tail of k_pt_swap which is run here",
    "k_copy_strided_f64": "strided copy",
    "k_transpose_hist_f64": "strided copy",
    "k_xor_words": "a ^= b",
}


def test_every_kernel_is_run_here_or_accounted_for():
    kernels = set()
    for name in os.listdir(CSRC):
        if name.endswith((".cu", ".cuh")):
            text = re.sub(r"//.*", "", open(os.path.join(CSRC, name)).read())
            kernels |= set(re.findall(r"__global__[^;{]*?\b(k_\w+)\s*\(", text, flags=re.S))
    assert len(kernels) >= 35, sorted(kernels)
    run_here = set()
    for name in os.listdir(EMU):
        if name.endswith(".cpp"):
            text = re.sub(r"//.*", "", open(os.path.join(EMU, name)).read())
            run_here |= set(re.findall(r"\b(k_\w+)\b", text))
    missing = kernels - run_here - set(NOT_EMULATED)
    assert not missing, f"kernels neither emulated nor accounted for: {sorted(missing)}"
    stale = (set(NOT_EMULATED) | run_here) - kernels
    assert not stale, f"names that are no kernels of the library (any more): {sorted(stale)}"
    assert not (set(NOT_EMULATED) & run_here)


# ---- the build-time variants of the row walk (A/B knobs of sweep_rows.cuh) give the same bits ------------------
VARIANTS = ["-DISING_ROWS_ZSKIP=1", "-DISING_ROWS_DEFER_RARE=0", "-DISING_ROWS_DEFER_RARE=1", "-DISING_ROWS_LT_SEL=1",
            "-DISING_ROWS_MUL_SPLIT=0"]


def test_row_walk_build_variants_give_the_same_bits(emu, oracle, tmp_path):
    """Every opt-in formulation kept in the source behind a macro (leading zero planes without the class
    select, the three placements of the rare tie path, ISETP/SEL tie compare, unsplit Philox products) is
    compiled for the host and must land on the mirror's bits like the default build - at a low and at a
    high inverse temperature (where all six threshold planes of a class are zero and ties are frequent)."""
    import shutil

    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    build = str(tmp_path)
    prepare_sources(os.path.join(build, "prepared"))
    procs = []
    for k, flag in enumerate(VARIANTS):
        so = os.path.join(build, f"variant{k}.so")
        procs.append((flag, so, subprocess.Popen(
            ["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-pthread", "-w", flag, "-I", EMU, "-I", build, "-I", cuda_inc,
             os.path.join(EMU, "emu_rows.cpp"), "-o", so], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    rng = np.random.default_rng(5)
    dims, E, W, V = (8, 4, 4), 128, 4, 4
    a, b, j = torus(dims, rng, True, -1.0)
    N = 128
    _, colors = layout_index(dims)
    init = rng.integers(0, 2, size=(E, N)).astype(bool)
    jm8 = bond_masks(dims, a, b, j)
    betas, seed = [0.1, 1.2, 2.0], 0x7A21A275
    en_ref, st_ref = oracle.msc_mirror(a, b, j, N, colors, E, seed, betas, states=init, per_sweep=True)
    for flag, so, pr in procs:
        _, err = pr.communicate()
        assert pr.returncode == 0, flag + ":\n" + err[-3000:]
        lib = C.CDLL(so)
        lib.emu_rows_phase.restype = C.c_int
        lib.emu_rows_phase.argtypes = emu.emu_rows_phase.argtypes
        for small in (0, 1):
            words = pack(init, dims, W)
            ens = []
            for s_, beta in enumerate(betas):
                for colour in (0, 1):
                    nsat = np.zeros(W * 32, dtype=np.uint64)
                    rc = lib.emu_rows_phase(3, dims[0], dims[1], dims[2], W, V, jm8.ctypes.data, 0, words.ctypes.data, colour,
                                            seed, s_, 0, float(beta), 1.0, int(colour == 1), nsat.ctypes.data, small, 3)
                    assert rc == 0, (flag, rc)
                ens.append(len(a) - 2.0 * nsat[:E].astype(np.float64))
            assert (unpack(words, dims, E) == st_ref).all(), flag
            assert (np.array(ens).T == en_ref).all(), flag


@pytest.mark.parametrize("Lx,Ly,nbands,j", [(256, 16, 3, -1.0), (512, 10, 5, 1.0), (256, 8, 1, -1.0)])
def test_fused_strip_pass_equals_the_mirror(emu, oracle, Lx, Ly, nbands, j):
    """k_strip_sweep_fused (opt-in): both colours of a sweep in one out-of-place pass over bands of rows with
    redundantly recomputed boundary rows - the same bits as two colour phases, hence as the mirror."""
    rng = np.random.default_rng(Lx + Ly + nbands)
    Wr, G = Lx // 64, 2
    init = rng.integers(0, 2, size=(Ly, Lx)).astype(bool)
    betas, seed = [0.35, 0.6, 0.9], 0x0DDBA11
    cur = np.zeros((2, Ly + 2 * G, Wr), dtype=np.uint32)
    cur[:, G:-G] = strip_pack(init, Wr)
    for t, beta in enumerate(betas):
        for c in range(2):                                        # periodic ghost rows of the source
            cur[c, :G] = cur[c, Ly:Ly + G]
            cur[c, -G:] = cur[c, G:2 * G]
        nxt = np.zeros_like(cur)
        rc = emu.emu_strip_fused(cur.ctypes.data, nxt.ctypes.data, Wr, Ly, 0, Ly, G, t, seed, 0xFFFFFFFF if j > 0 else 0,
                                 float(beta), abs(j), G - 1, Ly + 2, nbands)
        assert rc == 0
        cur = nxt
    got = strip_unpack(cur[:, G:-G], Lx)
    _, ref = oracle.msc_mirror_single(Lx, Ly, j, seed, betas, state=init)
    assert (got == ref).all()
