import os, sys, json, base64, ctypes, random
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle
L = ctypes.CDLL(os.path.join(HERE, 'libemu_dense.so'))
L.emu_count_dense.restype = ctypes.c_int64
L.emu_count_dense.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]

def emu(data, kmax, min_rec, tpt, tps, base_off):
    a = np.frombuffer(data, np.uint8) if len(data) else np.zeros(0, np.uint8)
    out = np.zeros(sum(4**j for j in range(1,kmax+1)), np.uint64)
    w = L.emu_count_dense(a.ctypes.data if a.size else None, a.size, base_off, kmax, min_rec, tpt, tps, out.ctypes.data, None)
    res, off = {}, 0
    for j in range(1,kmax+1):
        res[j] = out[off:off+4**j]; off += 4**j
    return res, w

def check(data, kmax, min_rec, tpt, tps, base_off, tag):
    res, w = emu(data, kmax, min_rec, tpt, tps, base_off)
    ok = True
    for j in range(1,kmax+1):
        ref = oracle.count_dense(data, j, min_rec)
        if not np.array_equal(ref, res[j]):
            ok = False
            d = np.nonzero(ref != res[j])[0]
            print('MISMATCH', tag, 'level', j, 'kmax', kmax, 'min_rec', min_rec, 'geom', tpt, tps, base_off, 'bins', [(oracle.code_to_kmer(b,j), int(ref[b]), int(res[j][b])) for b in d[:5]])
            break
    return ok

rng = random.Random(7)
cases = json.load(open(os.path.join(os.path.dirname(HERE), 'golden', 'extract_cases.json')))
nbad = 0; n=0
for c in cases:
    data = base64.b64decode(c['fasta_b64'])
    for kmax in (1,2,3,5,8,10):
        for trial in range(3):
            tpt = rng.choice([1,2,3,4,8]); tps = rng.choice([1,2,5]); bo = rng.choice([0,0,1,17,63,64,100])
            mr = kmax if trial<2 else kmax + rng.randint(1,9)
            n+=1
            if not check(data, kmax, mr, tpt, tps, bo, c['name']): nbad+=1
print('golden-derived checks', n, 'bad', nbad)

def rand_fasta(rng):
    parts=[]
    if rng.random()<0.2: parts.append(rng.choice(["junk\n","\n","ACGT\n; x\n"," >notheader\n"]))
    for r in range(rng.randint(0,6)):
        eol = rng.choice(["\n","\n","\r\n","\r"])
        parts.append(">" + "".join(rng.choice("ACGT>x y\t") for _ in range(rng.randint(0,150))) + eol)
        L_ = rng.choice([0,1,2,5,11,12,13,rng.randint(0,400),rng.randint(0,400)])
        alpha = rng.choice(["ACGT","ACGT","ACGTN","ACGTacgtnNRY>-","AC","ACGT \t"])
        seq = "".join(rng.choice(alpha) for _ in range(L_))
        if rng.random()<0.3:
            # N runs
            i = rng.randint(0,max(0,len(seq)-1)); seq = seq[:i] + "N"*rng.randint(1,40) + seq[i:]
        width = rng.choice([1,2,3,7,60,61,63,64,65,80,10**6])
        for i in range(0,len(seq),width):
            line = seq[i:i+width]
            if rng.random()<0.15: line += rng.choice([" ","\t"," \t ","\x0b","\x0c","\x1c"])
            parts.append(line+eol)
        if rng.random()<0.2: parts.append(eol*rng.randint(1,3))
    t = "".join(parts)
    if rng.random()<0.3: t = t.rstrip("\r\n")
    return t.encode('latin-1')

for it in range(1500):
    data = rand_fasta(rng)
    kmax = rng.choice([1,2,3,4,6,8,9,12])
    mr = kmax if rng.random()<0.75 else kmax+rng.randint(1,12)
    tpt = rng.choice([1,2,3,4,8,16]); tps = rng.choice([1,2,3,100]); bo = rng.choice([0,0,3,31,64,77])
    n+=1
    if not check(data, kmax, mr, tpt, tps, bo, 'fuzz%d'%it):
        nbad+=1
        if nbad>5: break
print('total checks', n, 'bad', nbad)
