"""The legacy boundary is a drop-in: the reference's OWN translation units compile, unchanged, against
include/legacy/*.cuh (same-named stand-ins for dev/*.cuh) and link with libunet_b200.so.

CPU suite, needs nvcc; every test but the struct-layout one also needs the reference's source tree.  The .cu file is
compiled from a scratch copy so that `#include "x.cuh"` resolves to include/legacy/x.cuh instead of the header
beside the source; dev/common.h / dev/rand.h / dev/common.cu (the reference's test infrastructure: validate_result,
fopenCheck, ...) are taken from the reference as they are.  Nothing is executed here (no GPU); the linked programs are
run on the B200 by tests/test_reference_cuda_gpu.py::test_legacy_programs_run.
"""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
NVCC = shutil.which("nvcc")

pytestmark = pytest.mark.skipif(not NVCC, reason="needs nvcc")
needs_reference = pytest.mark.skipif(not os.path.isdir(REF), reason="needs the reference's source tree")


def _nvcc(args, cwd):
    r = subprocess.run([NVCC, "-arch=sm_100", "-w", "-std=c++17"] + args, cwd=cwd, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]


@needs_reference
@pytest.mark.parametrize("name,layers_only", [("resblock", True), ("attention_block", True), ("unet_test", False)])
def test_reference_translation_unit_compiles_against_legacy_headers(tmp_path, name, layers_only):
    src = tmp_path / f"{name}.cu"
    shutil.copy(os.path.join(REF, "dev", f"{name}.cu"), src)
    # the source is byte-identical to the reference's
    assert open(src, "rb").read() == open(os.path.join(REF, "dev", f"{name}.cu"), "rb").read()
    args = ["-c", "-I", os.path.join(ROOT, "include", "legacy"), "-I", os.path.join(REF, "dev"), str(src), "-o",
            str(tmp_path / f"{name}.o")]
    if layers_only:  # these files DEFINE resblock_* / attention_block_* on top of the layer API
        args.insert(0, "-DUB_LEGACY_LAYERS_ONLY")
    _nvcc(args, str(tmp_path))
    assert os.path.getsize(tmp_path / f"{name}.o") > 0


@needs_reference
def test_reference_programs_link_with_the_library(tmp_path, ub):
    """dev/resblock.cu (its own composites over OUR layer launchers) and dev/unet_test.cu (OUR composites) link."""
    libdir = os.path.dirname(ub.LIB_PATH)
    for name, layers_only in (("resblock", True), ("unet_test", False)):
        src = tmp_path / f"{name}.cu"
        shutil.copy(os.path.join(REF, "dev", f"{name}.cu"), src)
        args = (["-DUB_LEGACY_LAYERS_ONLY"] if layers_only else []) + [
            "-I", os.path.join(ROOT, "include", "legacy"), "-I", os.path.join(REF, "dev"), str(src),
            os.path.join(REF, "dev", "common.cu"), "-o", str(tmp_path / name), "-L", libdir, "-lunet_b200", "-lcublas"]
        _nvcc(args, str(tmp_path))
        syms = subprocess.run(["nm", "-D", "--undefined-only", str(tmp_path / name)], stdout=subprocess.PIPE,
                              text=True).stdout
        # the layer launchers resolve to the C ABI of this library
        assert "ub_conv2d_k3_forward3" in syms and "ub_groupnorm_forward" in syms
        if not layers_only:
            assert "ub_resblock_forward" in syms and "ub_attention_block_backward" in syms


def test_legacy_header_keeps_the_reference_struct_layouts(tmp_path):
    """sizeof / offsetof of every struct of dev/*.cuh, printed by a tiny probe compiled against the legacy header, equal
    the reference's layout stored in tests/golden/legacy_struct_layouts.txt, and the reference header's own probe output
    where the reference's tree is present.  The stored file is the legacy header's probe output from the commit where
    this test compared the two headers directly."""
    probe = r'''
#include <cstdio>
#include <cstddef>
#define P(T) std::printf(#T " %zu\n", sizeof(T))
#define O(T, f) std::printf(#T "." #f " %zu\n", offsetof(T, f))
int main() {
    P(ConvK3Params); P(ConvK3Acts); P(LinearParams); P(LinearActs); P(GroupNormParams); P(GroupNormActs);
    P(GroupNormBackActs); P(SiluActs); P(AvgpoolActs); P(UpsampleActs); P(ConcatChannelActs); P(TimestepEmbedding);
    P(ResBlockParameters); P(ResBlockActivations); P(ResBlockBackwardActivations);
    P(AttentionParams); P(AttentionActs); P(AttentionBackwardActs); P(AttentionConfig); P(AttentionDebugStates);
    O(ResBlockParameters, res_cv1_b); O(ResBlockParameters, param_sizes); O(ResBlockParameters, n_params);
    O(ResBlockActivations, add2); O(ResBlockActivations, act_sizes); O(ResBlockActivations, input); O(ResBlockActivations, emb);
    O(ResBlockBackwardActivations, demb); O(ResBlockBackwardActivations, back_sizes); O(ResBlockBackwardActivations, n_backs);
    O(AttentionParams, proj_b); O(AttentionParams, n_params); O(AttentionActs, add); O(AttentionActs, input);
    O(AttentionBackwardActs, dinp); O(AttentionBackwardActs, n_backs); O(GroupNormActs, rstd); O(TimestepEmbedding, max_period);
    std::printf("convk3 %zu linear %zu\n", convk3_count_params(192, 64), linear_count_params(256, 64));
    return 0;
}
'''
    with open(os.path.join(ROOT, "tests", "golden", "legacy_struct_layouts.txt")) as f:
        outs = [f.read()]
    probes = [("ours", ["unet_b200_legacy.hpp"])]
    if os.path.isdir(REF):
        probes.append(("ref", ["conv2d_k3.cuh", "linear.cuh", "groupnorm.cuh", "silu.cuh", "avgpool.cuh", "upsample.cuh",
                               "concat_channel.cuh", "timestep_embedding.cuh", "resblock.cuh", "attention_block.cuh"]))
    for tag, incs in probes:
        d = tmp_path / tag
        d.mkdir()
        src = d / "probe.cu"
        src.write_text("".join(f'#include "{h}"\n' for h in incs) + probe)
        inc = os.path.join(REF, "dev") if tag == "ref" else os.path.join(ROOT, "include")
        _nvcc(["-I", inc, str(src), "-o", str(d / "probe"), "-cudart", "static"], str(d))
        outs.append(subprocess.run([str(d / "probe")], stdout=subprocess.PIPE, text=True, check=True).stdout)
    assert all(o == outs[0] for o in outs[1:]), "\n".join(outs)
