#!/usr/bin/env python3
"""Randomised cross-check of the host logic and the CPU oracle against the UNMODIFIED reference: random cjpeg switch
sets on random small images through (a) the reference's own cjpeg binary (oracle/_ref, so only where the reference was
available at build time) and (b) the cjpeg mirror + b200jpeg_validate + the oracle.  Test infrastructure.
usage: fuzz_vs_reference.py [seed] [cases] [--record FILE | --recorded FILE]      (exit status 1 if anything differs)
--record writes what the reference did with every case to FILE; --recorded takes the reference's side from such a file
instead of running the reference, so the check runs where the reference is absent."""
import argparse, hashlib, json, os, random, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
from oracle import oracle as O
import mozjpeg_b200 as mj
from mozjpeg_b200 import _abi as A


def cases(seed, n):
    """(width, height, image seed, switches) of the run's cases, in order."""
    rng=random.Random(seed)
    for it in range(n):
        w=rng.choice([1,7,8,16,17,33,64,100,131]); h=rng.choice([1,5,8,16,23,40,64,77])
        s=rng.randrange(1<<20)
        sw=[]
        prof=rng.choice(["", "-revert", "-baseline", "-fastcrush", "-progressive"])
        if prof=="-progressive": sw+=["-revert","-progressive"] if rng.random()<0.5 else ["-progressive"]
        elif prof: sw.append(prof)
        if rng.random()<0.8: sw+=["-quality",str(rng.choice([5,20,40,60,75,80,85,90,95,100]))]
        if rng.random()<0.5: sw+=["-sample",rng.choice(["1x1","2x1","1x2","2x2","3x1","4x2","2x2,1x1,2x2","1x1,2x1,1x1","4x1,2x1,1x1"])]
        if rng.random()<0.2: sw+=["-grayscale"]
        if rng.random()<0.25: sw+=["-restart",rng.choice(["1","2","3B","7B","1B"])]
        if rng.random()<0.2: sw+=["-dct",rng.choice(["fast","float","int"])]
        if rng.random()<0.15: sw+=["-smooth",str(rng.choice([1,10,50,100]))]
        if rng.random()<0.15: sw+=[rng.choice(["-notrellis","-notrellis-dc","-noovershoot","-optimize","-nojfif","-quant-baseline"])]
        if rng.random()<0.1: sw+=["-quant-table",str(rng.randrange(0,9))]
        if rng.random()<0.1: sw+=[rng.choice(["-tune-psnr","-tune-ssim","-tune-ms-ssim","-tune-hvs-psnr"])]
        if rng.random()<0.1: sw+=["-dc-scan-opt",str(rng.randrange(0,3))]
        if rng.random()<0.1: sw+=["-trellis-dc-ver-weight",rng.choice(["0.5","1.0","3"])]
        if rng.random()<0.1: sw+=["-lambda1",rng.choice(["9","12.5","14.75"]),"-lambda2",rng.choice(["0","13","16.5"])]
        yield w, h, s, sw


def reference(w, h, s, sw):
    """What the reference's cjpeg makes of a case: {"ok", "size", "md5"} or {"ok": False, "error"}."""
    try:
        a=O._ref_cjpeg_pixels(O.synth_image(s,w,h),sw)
    except Exception as ex:
        return {"ok": False, "error": str(ex).strip().splitlines()[-1][-70:]}
    return {"ok": True, "size": len(a), "md5": hashlib.md5(a).hexdigest()}


def main():
    ap=argparse.ArgumentParser()
    ap.add_argument("seed", type=int, nargs="?", default=1)
    ap.add_argument("cases", type=int, nargs="?", default=150)
    g=ap.add_mutually_exclusive_group()
    g.add_argument("--record", metavar="FILE")
    g.add_argument("--recorded", metavar="FILE")
    args=ap.parse_args()
    todo=list(cases(args.seed, args.cases))
    if args.recorded:
        rec=json.load(open(args.recorded))
        if rec["seed"]!=args.seed or len(rec["cases"])<len(todo):
            sys.exit(f"{args.recorded} holds seed {rec['seed']}, {len(rec['cases'])} cases: not this run's")
        refs=rec["cases"][:len(todo)]
        for (w,h,s,sw),r in zip(todo,refs):
            if [r["width"],r["height"],r["seed"],r["switches"]]!=[w,h,s,sw]:
                sys.exit(f"{args.recorded} does not hold the cases this generator makes (first difference: {sw})")
    else:
        refs=[reference(*c) for c in todo]
    if args.record:
        json.dump({"generator": "tools/fuzz_vs_reference.py --record", "seed": args.seed,
                   "cases": [dict(width=w, height=h, seed=s, switches=sw, **r) for (w,h,s,sw),r in zip(todo,refs)]},
                  open(args.record,"w"), indent=0)
    lib=A.load()
    bad=0; tot=0; refused=0
    for (w,h,s,sw),r in zip(todo,refs):
        ref_ok=r["ok"]
        try:
            p=mj.params_from_switches(sw,w,h,3)
        except Exception as ex:
            if ref_ok: print("MIRROR REJECTS what reference accepts:",sw,ex); bad+=1
            continue
        rc=lib.b200jpeg_validate(C.byref(p))
        if not ref_ok:
            if rc==0: print("WE ACCEPT what reference rejects:",sw,(w,h),r["error"]); bad+=1
            continue
        if rc!=0:
            refused+=1
            if rc==-1: print("WE REJECT (PARAM) what reference accepts:",sw,(w,h),lib.b200jpeg_last_error()); bad+=1
            continue
        tot+=1
        try: b=O.oracle_encode(p,O.synth_image(s,w,h)).jpeg
        except Exception as ex: print("ORACLE FAIL",sw,(w,h),ex); bad+=1; continue
        if (len(b),hashlib.md5(b).hexdigest())!=(r["size"],r["md5"]): bad+=1; print("MISMATCH",sw,(w,h),r["size"],len(b))
    print("seed", args.seed, "cases", args.cases, "bad", bad, "compared", tot, "refused(unsupported)", refused)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
