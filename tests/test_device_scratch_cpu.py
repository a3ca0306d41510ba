"""Device memory ownership of the CUDA sources, checked without a GPU.

Every per-call device buffer is taken through asp_scratch::get (csrc/common.cuh) and given back by the owner, so an early
return cannot leak stream-ordered memory.  Raw cudaMallocAsync / cudaFreeAsync calls are allowed only in the owner itself
and in the functions that fill or free the long-lived handles (space, graph, the graph's lambda-pass blob)."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pyarrowspace_b200", "csrc")

# function -> what its cudaMallocAsync may fill (the first argument)
MALLOC_ALLOWED = {
    "asp_scratch": r"&p\b",                    # get()
    "asp_space_create": r"&s->",               # the space's items, norms, lambdas
    "asp_space_adopt_shard": r"&s->",
    "asp_graph_from_csr": r"&g->",             # the stored Laplacian
    "asp_assemble_laplacian": r"&g->",         # the Laplacian CSR of a new graph
    "build_tm_blob": r"&out->",                # the graph's lambda-pass inputs
    "knn_row_norms": r"&s->nsq\b",             # the space's sums of squares
}
# functions that may call cudaFreeAsync: the owner and the handle free functions
FREE_ALLOWED = {"asp_scratch", "asp_free_space", "asp_free_graph", "asp_graph_free_upper"}

_SKIP_FIRST = " \t/#{}"


def _code_lines(path):
    """Source lines with // comments removed (the sources keep no '//' inside string literals)."""
    with open(path) as fh:
        return [re.sub(r"//.*", "", line.rstrip("\n")) for line in fh]


def _enclosing(lines, i):
    """Name of the function or struct whose definition encloses line i: the nearest line above that starts in column 0."""
    for line in reversed(lines[: i + 1]):
        if not line or line[0] in _SKIP_FIRST or line.startswith(("extern", "namespace", "template")):
            continue
        m = re.match(r"(?:struct|class)\s+(\w+)", line)
        if m:
            return m.group(1)
        m = re.search(r"(\w+)\s*\(", line)
        if m:
            return m.group(1)
    return None


def scan(csrc=CSRC):
    """(violations, owner_sites): every raw allocation or free outside the allow-lists, and how many the owner has."""
    bad, owner = [], 0
    for path in sorted(glob.glob(os.path.join(csrc, "*.cu*"))):
        lines = _code_lines(path)
        name = os.path.basename(path)
        for i, line in enumerate(lines):
            for m in re.finditer(r"\bcuda(Malloc|Free)Async\s*\(\s*([^,]*)", line):
                kind, arg = m.group(1), m.group(2)
                fn = _enclosing(lines, i)
                where = f"{name}:{i + 1} in {fn}: {line.strip()}"
                if fn == "asp_scratch":
                    owner += 1
                if kind == "Free":
                    if fn not in FREE_ALLOWED:
                        bad.append("cudaFreeAsync outside the owner: " + where)
                elif fn not in MALLOC_ALLOWED or not re.match(MALLOC_ALLOWED[fn], arg):
                    bad.append("cudaMallocAsync outside the owner: " + where)
    return bad, owner


def test_device_buffers_have_one_owner():
    bad, owner = scan()
    assert owner == 2, "asp_scratch should hold the one cudaMallocAsync (get) and the one cudaFreeAsync (release)"
    assert not bad, f"{len(bad)} raw stream-ordered allocation site(s); take the buffer with asp_scratch::get:\n" + "\n".join(bad)


def test_scan_finds_enclosing_functions():
    lines = [
        "static int helper(int a,",
        "                  int b)",
        "{",
        "    cudaFreeAsync(p, st);   ",
        "}",
        "struct Owner {",
        "    void release() { for (void *p : ptrs) cudaFreeAsync(p, st); }",
        "};",
    ]
    assert _enclosing(lines, 3) == "helper"
    assert _enclosing(lines, 6) == "Owner"
