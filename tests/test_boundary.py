"""CPU: the drop-in boundary claim of INTEGRATION.md section 2, checked against the reference's own adapter source.

A temporary copy of racon's src/cuda/cudabatch.{hpp,cpp} receives ONLY the textual changes INTEGRATION.md
shows (include of the shim, the cudapoa namespace) and must then compile (`g++ -fsyntax-only -DCUDA_ENABLED`)
against racon_gpu_b200/csrc/host/b200poa_batch.hpp -- racon's adapter is the FFI of this path, so this is the
"binding builds" check.  racon's sources are taken where oracle/Makefile builds the reference from (its REF, which
the environment can override); skipped where they are not present."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = subprocess.run(["make", "-s", "--no-print-directory", "-C", os.path.join(ROOT, "oracle"), "print-ref"],
                     capture_output=True, text=True).stdout.strip()
NO_SOURCES = not (REF and os.path.isdir(os.path.join(REF, "src", "cuda")))


@pytest.mark.skipif(NO_SOURCES, reason="racon's sources not present (oracle/Makefile REF)")
@pytest.mark.parametrize("shim_first", [False, True])
def test_racons_cudabatch_builds_against_the_shim_with_the_documented_diff(tmp_path, shim_first):
    for f in ("cudabatch.hpp", "cudabatch.cpp"):
        shutil.copy(os.path.join(REF, "src", "cuda", f), tmp_path / f)
        os.chmod(tmp_path / f, 0o644)
    hpp = (tmp_path / "cudabatch.hpp").read_text()
    assert "#include <claraparabricks/genomeworks/cudapoa/batch.hpp>" in hpp
    hpp = hpp.replace("#include <claraparabricks/genomeworks/cudapoa/batch.hpp>", '#include "b200poa_batch.hpp"')
    hpp = hpp.replace("std::unique_ptr<claraparabricks::genomeworks::cudapoa::Batch> cudapoa_batch_;",
                      "std::unique_ptr<b200poa_cpp::Batch> cudapoa_batch_;")
    (tmp_path / "cudabatch.hpp").write_text(hpp)
    cpp = (tmp_path / "cudabatch.cpp").read_text()
    assert "using namespace claraparabricks::genomeworks::cudapoa;" in cpp
    cpp = cpp.replace("using namespace claraparabricks::genomeworks::cudapoa;", "using namespace b200poa_cpp;")
    (tmp_path / "cudabatch.cpp").write_text(cpp)
    shim = ["-I", os.path.join(ROOT, "racon_gpu_b200", "csrc", "host"), "-I", os.path.join(ROOT, "include")]
    racon = ["-I", os.path.join(REF, "src"), "-I", os.path.join(REF, "src", "cuda")]
    inc = (shim + racon) if shim_first else (racon + shim)  # either order: nothing of ours shadows racon's headers
    cmd = ["g++", "-std=c++14", "-fsyntax-only", "-DCUDA_ENABLED", "-I", str(tmp_path), *inc,
           "-I", os.path.join(REF, "vendor", "spoa", "include"),
           "-I", os.path.join(REF, "vendor", "GenomeWorks", "common", "base", "include"),  # GW_CU_CHECK_ERR only
           "-I", os.path.join(REF, "vendor", "GenomeWorks", "3rdparty", "spdlog", "include"),
           "-I", "/usr/local/cuda/include", str(tmp_path / "cudabatch.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]


@pytest.mark.skipif(NO_SOURCES, reason="racon's sources not present (oracle/Makefile REF)")
def test_racons_cudaaligner_builds_against_the_shim_with_the_documented_diff(tmp_path):
    """INTEGRATION.md section 5: racon's CUDABatchAligner (src/cuda/cudaaligner.{hpp,cpp}) over b200aln_aligner.hpp."""
    for f in ("cudaaligner.hpp", "cudaaligner.cpp"):
        shutil.copy(os.path.join(REF, "src", "cuda", f), tmp_path / f)
        os.chmod(tmp_path / f, 0o644)
    hpp = (tmp_path / "cudaaligner.hpp").read_text()
    for inc in ("cudaaligner.hpp", "aligner.hpp", "alignment.hpp"):
        line = "#include <claraparabricks/genomeworks/cudaaligner/%s>" % inc
        assert line in hpp
        hpp = hpp.replace(line, '#include "b200aln_aligner.hpp"' if inc == "aligner.hpp" else "")
    assert "std::unique_ptr<claraparabricks::genomeworks::cudaaligner::Aligner> aligner_;" in hpp
    hpp = hpp.replace("std::unique_ptr<claraparabricks::genomeworks::cudaaligner::Aligner> aligner_;",
                      "std::unique_ptr<b200aln_cpp::Aligner> aligner_;")
    (tmp_path / "cudaaligner.hpp").write_text(hpp)
    cpp = (tmp_path / "cudaaligner.cpp").read_text()
    assert "using namespace claraparabricks::genomeworks::cudaaligner;" in cpp
    cpp = cpp.replace("using namespace claraparabricks::genomeworks::cudaaligner;", "using namespace b200aln_cpp;")
    (tmp_path / "cudaaligner.cpp").write_text(cpp)
    cmd = ["g++", "-std=c++14", "-fsyntax-only", "-DCUDA_ENABLED", "-I", str(tmp_path),
           "-I", os.path.join(REF, "src"), "-I", os.path.join(REF, "src", "cuda"),
           "-I", os.path.join(ROOT, "racon_gpu_b200", "csrc", "host"), "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(REF, "vendor", "GenomeWorks", "common", "base", "include"),  # GW_CU_CHECK_ERR only
           "-I", os.path.join(REF, "vendor", "GenomeWorks", "3rdparty", "spdlog", "include"),
           "-I", "/usr/local/cuda/include", str(tmp_path / "cudaaligner.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
