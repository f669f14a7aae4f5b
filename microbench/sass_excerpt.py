"""Per-kernel SASS instruction census of the in-tree library (no GPU needed):
    python microbench/sass_excerpt.py > profiles/r2_sass_excerpt.txt"""
import collections, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = os.path.join(ROOT, 'sdrterm_b200', 'libsdrterm_b200.so')
out = subprocess.run(['cuobjdump', '-sass', so], capture_output=True, text=True).stdout
WANT = ['UTCIMMA', 'UTCBAR', 'LDTM', 'UTMALDG', 'UTMAPF', 'SYNCS', 'DMMA', 'DFMA', 'DADD', 'DMUL', 'F2F', 'IMAD', 'LDS', 'STS',
        'SHFL', 'LDG', 'STG', 'LDGSTS', 'MUFU']
KEEP = ('k_tc', 'k_main', 'k_finish', 'k_fixup', 'k_demod', 'k_iqgain', 'k_iqtiles', 'k_iqscan_c', 'k_iqchunk', 'k_savgol', 'k_gfft4',
        'k_gfft2', 'k_spectrum_db', 'k_stft_db', 'k_decode', 'k_correct_iq')
print('# cuobjdump -sass sdrterm_b200/libsdrterm_b200.so (microbench/sass_excerpt.py): Blackwell-native instructions per kernel')
print('# UTCIMMA = tcgen05.mma.kind::i8, LDTM = tcgen05.ld, UTMALDG = TMA tensor load, UTMAPF = TMA L2 prefetch,')
print('# UTCBAR = tcgen05.commit, SYNCS = mbarrier, DMMA = FP64 tensor pipe (mma.sync.m8n8k4.f64), DFMA = FP64 FMA')
print('# (one instantiation per kernel template is listed: the int16 one, ENC = 2, where there is a choice)\n')
cur, cnt, seen = None, None, set()


def flush():
    if cur is None:
        return
    base = re.sub(r'^_Z\d+', '', cur)
    name = next((k for k in KEEP if base.startswith(k)), None)
    if name is None:
        return
    key = name
    if 'ILi' in cur and 'ILi2E' not in cur and name not in ('k_tc',):
        return
    if name == 'k_tc':
        key = cur
    if key in seen:
        return
    seen.add(key)
    tot = sum(cnt.values())
    print(cur)
    print(f'   total {tot} instr; ' + ', '.join(f'{k} {cnt[k]}' for k in WANT if cnt.get(k)))


for line in out.splitlines():
    m = re.match(r'\s*Function : (\S+)', line)
    if m:
        flush()
        cur, cnt = m.group(1), collections.Counter()
        continue
    m = re.match(r'\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)', line)
    if m and cur:
        cnt[m.group(1).split('.')[0]] += 1
        cnt['_all'] += 0
flush()
