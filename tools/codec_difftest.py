"""Differential test of the JPEG coefficient codec (csrc/jpegcoef.c) on random files: Pillow writes JPEGs of
random size / quality / sub-sampling / Huffman optimisation / restart intervals / progressive mode, and the
lossless transcode (`jpegqs -n 0`) must give the same bytes with the one-thread reader, with the threaded
reader (random thread count and chunk size) and with the reference's own quantsmooth.c on libjpeg-turbo
(oracle/_ref/refcli_cpu, built by oracle/Makefile).  No GPU needed.
    python tools/codec_difftest.py [seed] [files]      (in a scratch directory: it writes in.jpg, s.jpg, p.jpg, r.jpg)
    python tools/codec_difftest.py seed files DIGESTS  (refcli_cpu's files given as their SHA-256 in the JSON file
                                                        DIGESTS, {file number: digest}; refcli_cpu is not run)
    python tools/codec_difftest.py seed files --record (also prints that JSON as the last line)
Round 2: seeds 1-3, 800 files, 0 mismatches."""
import hashlib, json, os, subprocess, sys, numpy as np
from PIL import Image
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E=os.path.join(ROOT,"jpeg-quantsmooth_b200","csrc","jpegqs"); R=os.path.join(ROOT,"oracle","_ref","refcli_cpu")
rng=np.random.RandomState(int(sys.argv[1]) if len(sys.argv)>1 else 1)
N=int(sys.argv[2]) if len(sys.argv)>2 else 200
record=len(sys.argv)>3 and sys.argv[3]=="--record"
stored=json.load(open(sys.argv[3])) if len(sys.argv)>3 and not record else None
digests={}
bad=0
for it in range(N):
    w=int(rng.randint(8,900)); h=int(rng.randint(8,700)); gray=rng.rand()<0.2
    kind=rng.randint(4)
    y,x=np.mgrid[0:h,0:w]
    base=128+rng.randint(10,90)*np.sin(x/rng.uniform(3,80))+rng.randint(10,60)*np.cos(y/rng.uniform(3,80))
    noise=rng.normal(0,rng.choice([0.5,3,10,40]),(h,w,3))
    img=(np.stack([base,base[::-1],base[:,::-1]],-1)+noise).clip(0,255).astype(np.uint8)
    im=Image.fromarray(img,"RGB")
    if gray: im=im.convert("L")
    kw=dict(quality=int(rng.choice([1,5,20,50,75,90,95,100])))
    if not gray: kw["subsampling"]=int(rng.randint(3))
    if rng.rand()<0.3: kw["optimize"]=True
    r=rng.rand()
    if r<0.25: kw["restart_marker_rows"]=int(rng.randint(1,5))
    elif r<0.5: kw["restart_marker_blocks"]=int(rng.randint(1,40))
    if rng.rand()<0.15: kw["progressive"]=True
    try:
        im.save("in.jpg",**kw)
    except OSError:
        continue
    env=dict(os.environ,JPEGQS_SERIAL_DECODE="1",JPEGQS_CODEC_THREADS="1")
    assert subprocess.run([E,"-n","0","-i","0","in.jpg","s.jpg"],env=env).returncode==0,(it,kw)
    th=str(int(rng.randint(4,17))); mb=str(int(rng.choice([64,300,2000,20000])))
    env=dict(os.environ,JPEGQS_CODEC_THREADS=th,JPEGQS_PAR_MIN_BYTES=mb,JPEGQS_CODEC_TRACE="1")
    p=subprocess.run([E,"-n","0","-i","0","in.jpg","p.jpg"],env=env,capture_output=True,text=True)
    assert p.returncode==0,(it,kw,p.stderr)
    a,b=(open(f,"rb").read() for f in ("s.jpg","p.jpg"))
    if stored is None:
        assert subprocess.run([R,"-n","0","-i","0","in.jpg","r.jpg"]).returncode==0
        digests[str(it)]=hashlib.sha256(open("r.jpg","rb").read()).hexdigest()
    else:
        digests[str(it)]=stored[str(it)]
    c=hashlib.sha256(a).hexdigest()==digests[str(it)]
    if not (a==b and c):
        bad+=1; print("MISMATCH",it,w,h,gray,kw,th,mb,a==b,c); os.rename("in.jpg",f"bad{it}.jpg")
    if "abandoned" in p.stderr: print("abandoned:",it,kw,th,mb)
print("done",N,"bad",bad)
if record: print(json.dumps(digests))
sys.exit(1 if bad else 0)
