"""Static checks that stand in for a GPU on code paths the CPU suite cannot execute: every Python file parses, and no
function reads a name that nothing in the file binds (imports, definitions, assignments, arguments) - the NameError
class of bugs in CUDA-only branches."""
import ast
import builtins
import glob
import os

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), os.pardir))
SKIP = (os.sep + "baseline" + os.sep, os.sep + "_build" + os.sep, "gpurun_out", os.sep + ".git" + os.sep)


def _files():
    for f in glob.glob(os.path.join(ROOT, "**", "*.py"), recursive=True):
        if not any(s in f for s in SKIP):
            yield f


def test_every_python_file_parses_and_binds_the_names_it_reads():
    module_names = set(dir(builtins)) | {"__file__", "__name__", "__doc__", "__path__", "__spec__", "__package__"}
    problems = {}
    for path in _files():
        with open(path, errors="ignore") as f:
            tree = ast.parse(f.read(), filename=path)          # SyntaxError fails the test with the location
        bound, star = set(module_names), False
        for n in ast.walk(tree):
            if isinstance(n, (ast.FunctionDef, ast.AsyncFunctionDef, ast.ClassDef)):
                bound.add(n.name)
            elif isinstance(n, ast.Import):
                bound.update((a.asname or a.name).split(".")[0] for a in n.names)
            elif isinstance(n, ast.ImportFrom):
                star = star or any(a.name == "*" for a in n.names)
                bound.update(a.asname or a.name for a in n.names)
            elif isinstance(n, ast.Name) and isinstance(n.ctx, (ast.Store, ast.Del)):
                bound.add(n.id)
            elif isinstance(n, ast.arg):
                bound.add(n.arg)
            elif isinstance(n, ast.ExceptHandler) and n.name:
                bound.add(n.name)
            elif isinstance(n, (ast.Global, ast.Nonlocal)):
                bound.update(n.names)
            elif isinstance(n, ast.MatchAs) and n.name:
                bound.add(n.name)
        if star:
            continue
        read = {n.id for n in ast.walk(tree) if isinstance(n, ast.Name) and isinstance(n.ctx, ast.Load)}
        missing = sorted(read - bound)
        if missing:
            problems[os.path.relpath(path, ROOT)] = missing
    assert not problems, problems


def test_every_args_attribute_is_a_flag_or_assigned_somewhere(monkeypatch):
    """``args.<name>`` read anywhere in the package / entry points / tasks must be a destination of one of the argument
    parsers or be assigned somewhere (the reference lost ``--bert_no_binary_head`` from its parser while
    pretrain_bert.py kept reading it: this is the check that would have caught it)."""
    import re
    import sys
    sys.path.insert(0, ROOT)
    monkeypatch.setenv("MLB200_FORCE_CPU", "1")
    import finetune
    from megatron_llm_b200.arguments import build_base_parser
    dests = {a.dest for a in finetune.extra_args(build_base_parser())._actions}
    for mod_name, fn_name in (("pretrain_bert", "extra_args"), ("pretrain_t5", "extra_args"),
                              ("pretrain_ict", "extra_args"), ("tasks.main", "get_tasks_args"),
                              ("tasks.msdp.main", "get_tasks_args"), ("verify_correctness", "extra_extra_args")):
        try:
            mod = __import__(mod_name, fromlist=[fn_name])
        except Exception:  # noqa: BLE001 - optional entry points
            continue
        if hasattr(mod, fn_name):
            dests |= {a.dest for a in getattr(mod, fn_name)(build_base_parser())._actions}
    files = [f for f in _files() if os.sep + "tests" + os.sep not in f and os.sep + "tools" + os.sep not in f
             and os.sep + "weights_conversion" + os.sep not in f]
    assigned, used = set(), {}
    for path in files:
        src = open(path, errors="ignore").read()
        assigned |= set(re.findall(r"\bargs\.([A-Za-z_]\w*)\s*(?:=[^=]|,\s*args\.)", src))
        assigned |= set(re.findall(r"args\.[A-Za-z_]\w*,\s*args\.([A-Za-z_]\w*)\s*(?:=[^=]|,)", src))
        assigned |= set(re.findall(r"""setattr\(args,\s*["'](\w+)["']""", src))
        guarded = set(re.findall(r"""(?:hasattr|getattr)\(args,\s*["'](\w+)["']""", src))
        for m in re.finditer(r"\bargs\.([A-Za-z_]\w*)", src):
            if m.group(1) not in guarded:
                used.setdefault(m.group(1), set()).add(os.path.relpath(path, ROOT))
    unknown = {k: sorted(v)[:3] for k, v in used.items() if k not in dests and k not in assigned}
    assert not unknown, unknown


def test_build_restores_the_reference_tree_of_the_benchmark_arm(tmp_path, monkeypatch):
    """``baseline/_ref`` (the unmodified reference that ``bench.py --impl reference`` drives) is git-ignored, so a
    fresh checkout lacks it: ``__graft_entry__.build()`` copies the checkout named by ``MLB200_REFERENCE_DIR`` there,
    verbatim, and leaves an existing one alone.  A small stand-in tree plays the reference checkout."""
    import filecmp
    import __graft_entry__ as entry
    src = tmp_path / "Megatron-LLM"
    for rel, text in [("megatron/__init__.py", ""), ("megatron/training.py", "def pretrain():\n    pass\n"),
                      ("megatron/core/tensor_parallel/layers.py", "class ColumnParallelLinear:\n    pass\n"),
                      ("finetune.py", "from megatron.training import pretrain\n"), (".git/HEAD", "ref: main\n"),
                      ("megatron/__pycache__/training.cpython-312.pyc", "stale")]:
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_text(text)
    monkeypatch.setattr(entry, "ROOT", str(tmp_path / "repo"))
    ref = tmp_path / "repo" / "baseline" / "_ref"
    monkeypatch.delenv("MLB200_REFERENCE_DIR", raising=False)
    entry._ensure_reference_tree()
    assert not ref.exists()
    monkeypatch.setenv("MLB200_REFERENCE_DIR", str(src))
    entry._ensure_reference_tree()
    assert (ref / "megatron" / "training.py").is_file() and (ref / "finetune.py").is_file()
    assert not (ref / ".git").exists() and not (ref / "megatron" / "__pycache__").exists()

    def same(cmp):
        return (not cmp.left_only and not cmp.right_only and not cmp.diff_files
                and all(same(sub) for sub in cmp.subdirs.values()))
    assert same(filecmp.dircmp(str(src / "megatron"), str(ref / "megatron"), ignore=["__pycache__"]))
    marker = ref / "finetune.py"
    marker.write_text("# kept")
    entry._ensure_reference_tree()
    assert marker.read_text() == "# kept"
