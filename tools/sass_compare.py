"""Compare the SASS of two builds of librd_env.so kernel by kernel: which kernels of the first build compile to different
instructions (or are missing) in the second, and which kernels are new.  k_dense's trailing CONV template argument
(0 = a dense layer) is added to the first build's names, so a build from before that argument compares too.

    cuobjdump -sass old/librd_env.so > old.sass; cuobjdump -sass racing_dreamer_b200/librd_env.so > new.sass
    python tools/sass_compare.py old.sass new.sass
"""
import re
import sys


def functions(path):
    out, cur = {}, None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
        elif cur is not None and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            cur.append(re.sub(r"\s+", " ", line.strip()))
    return out


def with_conv0(name):
    return re.sub(r"^(_Z7k_denseI(?:Li\d+E|Lb\dE){7})(Ev8GemmMaps)", r"\1Li0E\2", name)


def main(old_path, new_path):
    old, new = functions(old_path), functions(new_path)
    same, diff = 0, []
    for name, body in old.items():
        other = new.get(with_conv0(name))
        if other != body:
            diff.append(("missing" if other is None else "differs") + " " + name)
        else:
            same += 1
    for d in diff:
        print(d)
    added = sorted(set(new) - {with_conv0(n) for n in old})
    print(f"{same} of {len(old)} kernels identical; new kernels: {', '.join(added) or 'none'}")
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:3]))
