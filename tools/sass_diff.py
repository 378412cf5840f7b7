"""Compare the SASS of every function of two builds of libnestfit_b200.so, function by function.

  cuobjdump -sass OLD.so > old.sass
  cuobjdump -sass NEW.so > new.sass
  python tools/sass_diff.py old.sass new.sass

Names of anonymous namespaces (which carry a hash of the source path) are normalised, and in the new build the
hyperfine kernel's defaulted sixth template argument (MOM = false) is dropped, so that every function of the old
build is compared with its counterpart.  Prints the counts and the names of differing, missing and added functions;
exits 1 when a function of the old build differs or is missing."""
import argparse
import re
import sys


def parse(path):
    """{mangled name: SASS lines} of a cuobjdump -sass listing (the source-file identifier lines left out)."""
    funcs, cur = {}, None
    with open(path) as f:
        for line in f:
            if line.startswith("Fatbin"):
                cur = None
            m = re.match(r"\s*Function : (\S+)", line)
            if m:
                cur = m.group(1)
                funcs[cur] = []
                continue
            if cur is not None and line.strip() and not line.strip().startswith("identifier"):
                funcs[cur].append(line.rstrip())
    return funcs


def norm(name, after=False):
    """The name with the path hash of anonymous namespaces removed; `after`: also without the trailing MOM = false."""
    name = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_cu_[0-9a-f]+", r"_GLOBAL__N_\1", name)
    if after:
        name = re.sub(r"^(_Z13nf_nh3_kernelI(?:Li\d+E){2}Lb[01]E[fd]Lb[01]E)Lb0EEv", r"\1Ev", name)
    return name


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    args = ap.parse_args()
    old = {norm(k): v for k, v in parse(args.old).items()}
    new = {norm(k, True): v for k, v in parse(args.new).items()}
    same = [k for k in old if new.get(k) == old[k]]
    diff = [k for k in old if k in new and new[k] != old[k]]
    missing = [k for k in old if k not in new]
    added = [k for k in new if k not in old]
    print(f"{len(old)} functions before, {len(new)} after: {len(same)} identical, {len(diff)} differ, "
          f"{len(missing)} missing, {len(added)} added")
    for tag, names in (("DIFF", diff), ("MISSING", missing), ("ADDED", added)):
        for k in names:
            print(tag, k)
    return 1 if diff or missing else 0


if __name__ == "__main__":
    sys.exit(main())
