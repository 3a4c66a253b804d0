"""Compare the SASS of two builds of one kernel file, function by function.

    cuobjdump -sass old.o > old.sass ; cuobjdump -sass new.o > new.sass
    python scripts/sass_diff.py old.sass new.sass

Function names are demangled (cu++filt).  A kernel that gained a trailing template parameter keeps its identity when that
parameter is given with --extra (default: "(bool)1", cu++filt's spelling of true, the value of the instantiations that keep the previous behaviour):
``f<1, 3, true>`` in the new dump is compared with ``f<1, 3>`` in the old one.  Instructions are compared with their encodings;
only the address comments are dropped.  Prints one line per old function and exits non-zero if any differs or is missing."""
import argparse
import re
import subprocess
import sys


def functions(path):
    out, name = {}, None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
            continue
        if name is None:
            continue
        body = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).strip()       # address comment
        if body and not body.startswith("....."):
            out[name].append(body)
    return out


def demangle(names):
    if not names:
        return {}
    r = subprocess.run(["cu++filt"], input="\n".join(names), stdout=subprocess.PIPE, text=True, check=True)
    return dict(zip(names, r.stdout.splitlines()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--extra", default="(bool)1", help="value of the added trailing template parameter that keeps the old behaviour")
    a = ap.parse_args()
    old, new = functions(a.old), functions(a.new)
    dold, dnew = demangle(list(old)), demangle(list(new))
    by_name = {}
    for k, d in dnew.items():
        by_name[d] = k
        stripped = re.sub(r", %s>" % re.escape(a.extra), ">", d)
        if "<%s>" % a.extra in stripped:                                  # a kernel that was not a template before
            stripped = re.sub(r"^void ", "", stripped.replace("<%s>" % a.extra, ""))
        by_name.setdefault(stripped, k)
    bad = 0
    for k, d in sorted(dold.items(), key=lambda kv: kv[1]):
        nk = by_name.get(d)
        if nk is None:
            print("MISSING    %s" % d)
            bad += 1
        elif new[nk] == old[k]:
            print("identical  %s  (%d instructions)" % (d, len(old[k])))
        else:
            diff = sum(1 for x, y in zip(old[k], new[nk]) if x != y) + abs(len(old[k]) - len(new[nk]))
            print("DIFFERENT  %s  (%d of %d lines)" % (d, diff, len(old[k])))
            bad += 1
    extra = sorted(set(dnew.values()) - set(dnew[by_name[d]] for d in dold.values() if d in by_name))
    for d in extra:
        print("new        %s" % d)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
