"""tests/golden/presets.json: the material presets of the reference's object menu, parsed from ITS source
(mainApp.cpp:1499-1597 of the checkout PTB_REFERENCE_DIR names: set_col_texture / set_col_specular / set_col_roughness per menu id)."""
import json
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))


def parse(path):
    src = open(path).read()
    out = {}
    for m in re.finditer(r"case ID_([A-Z_]+):[^\n]*\n(.*?)break;", src, re.S):
        name, body = m.group(1).lower(), m.group(2)
        t = re.search(r"set_col_texture\(Vector\(([^)]*)\)", body)
        s = re.search(r"set_col_specular\(Vector\(([^)]*)\)", body)
        r = re.search(r"set_col_roughness\(Vector\(([^)]*)\)", body)
        if t and s and r:
            ev = lambda g: [float(eval(x)) for x in g.group(1).split(",")]
            out[name] = {"Kd": ev(t), "Ks": ev(s), "Ne": ev(r)}
    return out


if __name__ == "__main__":
    import sys
    sys.path.insert(0, os.path.dirname(HERE))
    from oracles import reference_dir
    assert reference_dir(), "set PTB_REFERENCE_DIR to a checkout of the reference"
    json.dump(parse(os.path.join(reference_dir(), "mainApp.cpp")), open(os.path.join(HERE, "presets.json"), "w"), indent=1, sort_keys=True)
