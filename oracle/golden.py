"""TEST INFRASTRUCTURE ONLY -- reading and writing the golden fixtures under tests/golden/.

A fixture is an ``np.savez_compressed`` file.  An array that occurs under several names (the reference
returns identical fields for many of its settings) is stored once: ``_alias_names[i]`` is another name of
the stored array ``_alias_targets[i]``.  That keeps every fixture under 1 MB without dropping a value.
"""
import numpy as np


def save(path, arrays):
    """Write ``arrays`` (name -> array) to ``path``, each distinct array (dtype, shape and bytes) once."""
    first, keep, names, targets = {}, {}, [], []
    for name in sorted(arrays):
        a = np.asarray(arrays[name])
        key = (a.dtype.str, a.shape, a.tobytes())
        if key in first:
            names.append(name)
            targets.append(first[key])
        else:
            first[key] = name
            keep[name] = a
    np.savez_compressed(path, _alias_names=np.array(names, dtype=str), _alias_targets=np.array(targets, dtype=str),
                        **keep)


def load(path):
    """Every array of the fixture at ``path`` by name, aliases resolved (a dict of fresh arrays)."""
    with np.load(path) as z:
        g = {k: z[k] for k in z.files}
    for name, target in zip(g.pop("_alias_names", ()), g.pop("_alias_targets", ())):
        g[str(name)] = g[str(target)].copy()
    return g
