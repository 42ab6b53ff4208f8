"""Golden data for tests/test_integration_shim.py: what the reference's 3D/dcn/functions/deform_conv_func.py asks of the compiled
extension ``D3D`` -- the modules it imports ([module, name] for ``from module import name``) and, for every call into ``D3D``,
the calling method, the function name and the number of positional arguments -- read from the reference source with ``ast``.
Run where the reference tree is present:

    python tests/golden/make_golden_shim.py REFERENCE_ROOT        (writes tests/golden/ref3d_deform_conv_func.json)
"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref_root):
    tree = ast.parse(open(os.path.join(ref_root, "3D", "dcn", "functions", "deform_conv_func.py")).read())
    imports = []
    for node in ast.walk(tree):
        if isinstance(node, ast.Import):
            imports += [[a.name, None] for a in node.names]
        elif isinstance(node, ast.ImportFrom) and node.module != "__future__":
            imports += [[node.module, a.name] for a in node.names]
    calls = []
    for cls in (n for n in tree.body if isinstance(n, ast.ClassDef)):
        for fn in (n for n in cls.body if isinstance(n, ast.FunctionDef)):
            for node in ast.walk(fn):
                if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and isinstance(node.func.value, ast.Name)
                        and node.func.value.id == "D3D"):
                    assert not node.keywords and not any(isinstance(a, ast.Starred) for a in node.args)
                    calls.append({"caller": f"{cls.name}.{fn.name}", "function": node.func.attr, "positional_args": len(node.args)})
    path = os.path.join(HERE, "ref3d_deform_conv_func.json")
    with open(path, "w") as f:
        json.dump({"imports": imports, "d3d_calls": calls}, f, indent=1)
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    main(sys.argv[1])
