"""On-disk batch format (SURVEY.md section 8f-5; the reference has no wire / disk format at all).

One `.npz` file holds a batch of shared structure exactly as the engine consumes it, plus -- optionally -- the
results somebody obtained for it, so that benchmarks are reproducible and regression goldens travel:

    format            "sco_b200.batch"          version  1
    structure         JSON (n, stride, every Field as [off, shared], blocks, groups)  + the structure's arrays
                      (lin_rowptr / lin_col / lin_val, shared, group_overlap; st_cols<i>: column map of block i,
                      only for blocks that have one; st_ocols<i>: column map of objective block i)
    params [B, stride] float64      x0 [B, n] float64
    settings          JSON of the solver / OSQP settings the results belong to (optional)
    expected_*        verdict [B] int32, x [B, n], max_vio [B], objective [B], nonconverged [B] (optional)
    signature         sha256 of the structure (buckets of a mixed batch are files with different signatures)

    save_batch(path, st, params, x0, settings=None, expected=None)
    st, params, x0, meta = load_batch(path)
    python -m sco_py_b200.batchfile info  FILE        # what is inside
    python -m sco_py_b200.batchfile solve FILE        # solve on cuda:0, compare with expected_* if present
"""
import hashlib
import json
import sys

import numpy as np

from .structure import Block, Field, ObjBlock, Structure

FORMAT = "sco_b200.batch"
VERSION = 1
_FIELDS = ("Q", "q", "c", "lin_l", "lin_u", "obj_prog", "qa", "lb0", "ub0")
_ARRAYS = ("lin_rowptr", "lin_col", "lin_val", "shared", "group_overlap")


def _fld(f):
    return [int(f.off), bool(f.shared)]


def structure_to_json(st):
    d = dict(n=int(st.n), stride=int(st.stride), m_lin=int(st.m_lin), n_groups=int(st.n_groups),
             obj_prog_len=int(st.obj_prog_len), obj_prog_flags=int(st.obj_prog_flags))
    for name in _FIELDS:
        d[name] = _fld(getattr(st, name))
    d["blocks"] = [dict(family=int(b.family), cnt_type=int(b.cnt_type), m=int(b.m), par=_fld(b.par), val=_fld(b.val),
                        ipar=[int(v) for v in b.ipar], group_mask=int(b.group_mask), jw=int(b.jw)) for b in st.blocks]
    if st.obj_blocks:  # only when present: files and signatures of other structures stay as they were
        d["obj_blocks"] = [dict(prog=_fld(o.prog), m=int(o.m), n_in=int(o.n_in), n_instr=int(o.n_instr),
                                flags=int(o.flags)) for o in st.obj_blocks]
    return d


def _maps(st):
    """{array name: column map} of the blocks that have one."""
    maps = {"cols%d" % i: np.ascontiguousarray(b.cols, dtype=np.int32) for i, b in enumerate(st.blocks)
            if b.cols is not None}
    maps.update({"ocols%d" % i: np.ascontiguousarray(o.cols, dtype=np.int32) for i, o in enumerate(st.obj_blocks)})
    return maps


def structure_from_json(d, arrays):
    kw = {name: Field(int(d[name][0]), bool(d[name][1])) for name in _FIELDS if name in d}
    blocks = [Block(b["family"], b["cnt_type"], b["m"], Field(*b["par"]), Field(*b["val"]), ipar=list(b["ipar"]),
                    group_mask=b["group_mask"], jw=b["jw"], cols=arrays.get("cols%d" % i))
              for i, b in enumerate(d["blocks"])]
    for name in _ARRAYS:
        if name in arrays:
            kw[name] = arrays[name]
    kw["obj_blocks"] = [ObjBlock(Field(*o["prog"]), o["m"], o["n_in"], o["n_instr"], o["flags"], arrays["ocols%d" % i])
                        for i, o in enumerate(d.get("obj_blocks", []))]
    return Structure(n=d["n"], stride=d["stride"], m_lin=d["m_lin"], n_groups=d["n_groups"],
                     obj_prog_len=d.get("obj_prog_len", 0), obj_prog_flags=d.get("obj_prog_flags", 0), blocks=blocks, **kw)


def structure_signature(st):
    h = hashlib.sha256(json.dumps(structure_to_json(st), sort_keys=True).encode())
    for name in _ARRAYS:
        a = getattr(st, name)
        if a is not None:
            h.update(name.encode())
            h.update(np.ascontiguousarray(a).tobytes())
    for name, a in _maps(st).items():  # nothing for a structure without maps: its signature is unchanged
        h.update(name.encode())
        h.update(np.asarray(a.shape, dtype=np.int64).tobytes())
        h.update(a.tobytes())
    return h.hexdigest()


def save_batch(path, st, params, x0, settings=None, expected=None):
    params = np.ascontiguousarray(params, dtype=np.float64)
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    if params.shape != (x0.shape[0], st.stride) or x0.shape[1] != st.n:
        raise ValueError("params must be [B, %d] and x0 [B, %d]" % (st.stride, st.n))
    out = dict(format=np.array(FORMAT), version=np.array(VERSION), structure=np.array(json.dumps(structure_to_json(st))),
               signature=np.array(structure_signature(st)), params=params, x0=x0)
    for name in _ARRAYS:
        a = getattr(st, name)
        if a is not None:
            out["st_" + name] = np.asarray(a)
    for name, a in _maps(st).items():
        out["st_" + name] = a
    if settings is not None:
        out["settings"] = np.array(json.dumps(settings))
    for k, v in (expected or {}).items():
        out["expected_" + k] = np.asarray(v)
    np.savez_compressed(path, **out)


def load_batch(path):
    with np.load(path, allow_pickle=False) as z:
        if str(z["format"]) != FORMAT or int(z["version"]) > VERSION:
            raise ValueError("%s is not a %s file of version <= %d" % (path, FORMAT, VERSION))
        arrays = {k[3:]: z[k] for k in z.files if k.startswith("st_")}
        st = structure_from_json(json.loads(str(z["structure"])), arrays)
        if structure_signature(st) != str(z["signature"]):
            raise ValueError("%s: structure signature mismatch (file damaged or written by another version)" % path)
        meta = dict(signature=str(z["signature"]),
                    settings=json.loads(str(z["settings"])) if "settings" in z.files else None,
                    expected={k[len("expected_"):]: z[k] for k in z.files if k.startswith("expected_")})
        return st, z["params"], z["x0"], meta


def _main(argv):
    if len(argv) != 3 or argv[1] not in ("info", "solve"):
        print(__doc__)
        return 2
    st, params, x0, meta = load_batch(argv[2])
    print("%s: %d problems, n=%d m_lin=%d blocks=%s groups=%d stride=%d signature %s" % (
        argv[2], x0.shape[0], st.n, st.m_lin, [(b.family, b.m, b.cnt_type) for b in st.blocks], st.n_groups, st.stride,
        meta["signature"][:16]))
    print("settings:", meta["settings"], "| expected:", sorted(meta["expected"]))
    if argv[1] == "info":
        return 0
    from .engine import Engine, make_settings
    s = meta["settings"] or {}
    eng = Engine(st)
    out = eng.solve_batch_host(params, x0, make_settings(solver=s.get("solver"), osqp=s.get("osqp")))
    print("converged %d / %d" % (int((out["verdict"] == 1).sum()), x0.shape[0]))
    exp = meta["expected"]
    if "verdict" in exp:
        print("verdicts equal to the recorded ones: %d / %d" % (int((out["verdict"] == exp["verdict"]).sum()), x0.shape[0]))
    if "x" in exp:
        rel = np.abs(out["x"] - exp["x"]).max(axis=1) / np.maximum(1.0, np.abs(exp["x"]).max(axis=1))
        print("relative |dx| vs recorded: median %.2e max %.2e" % (float(np.median(rel)), float(rel.max())))
    return 0


if __name__ == "__main__":
    sys.exit(_main(sys.argv))
