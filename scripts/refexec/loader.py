"""Import the reference's model files by path under the paddle stand-in, without executing parakeet/__init__.py (which pulls
in librosa, visualdl, ... that are not installed): packages become empty namespace modules, modules load from their files."""
import importlib.abc
import importlib.util
import os
import sys
import types


class _RefFinder(importlib.abc.MetaPathFinder):
    def __init__(self, ref_root):
        self.ref_root = ref_root

    def find_spec(self, name, path=None, target=None):
        if name != "parakeet" and not name.startswith("parakeet."):
            return None
        rel = os.path.join(self.ref_root, *name.split("."))
        if os.path.isdir(rel):
            spec = importlib.util.spec_from_loader(name, loader=None, is_package=True)
            spec.submodule_search_locations = [rel]
            return spec
        if os.path.isfile(rel + ".py"):
            return importlib.util.spec_from_file_location(name, rel + ".py")
        return None


def install(standin_modules, ref_root):
    """Put the stand-in modules and a finder for the reference checkout at `ref_root` in place; returns an `uninstall()`."""
    saved = {k: sys.modules.get(k) for k in standin_modules}
    sys.modules.update(standin_modules)
    finder = _RefFinder(ref_root)
    sys.meta_path.insert(0, finder)

    def uninstall():
        sys.meta_path.remove(finder)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        for k in [k for k in sys.modules if k == "parakeet" or k.startswith("parakeet.")]:
            sys.modules.pop(k)
    return uninstall
