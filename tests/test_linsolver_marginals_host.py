"""CPU test of the LinearSolver-level marginal covariances (s3o_linsolver_solve_pattern): the declaration is valid C."""
import os
import subprocess

from conftest import ROOT


def test_linsolver_solve_pattern_declaration_compiles_as_c(tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "linsolver_marginals_snippet.c")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    "-c", src, "-o", str(tmp_path / "linsolver_marginals_snippet.o")], check=True)
