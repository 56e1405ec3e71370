import pathlib, sys; ROOT=pathlib.Path(__file__).resolve().parents[1]; sys.path.insert(0,str(ROOT))
import numpy as np, cv2
from svi_mapper_b200 import StereoFrontend, load_camera
from svi_mapper_b200.synth import stereo_pair
from oracle import frontend_np as o, c_oracle as co
cl=load_camera(str(ROOT/'tests/golden/calib/kitti_00_left.txt')); cr=load_camera(str(ROOT/'tests/golden/calib/kitti_00_right.txt'))
def variants(seed):
    L,R=stereo_pair(1241,376,seed)
    yield 'tex',L,R
    a=L.copy(); a[:120]=255; a[300:]=0; b=R.copy(); b[:120]=255; b[300:]=0
    yield 'sat',a,b
    yield 'post',(L//32*32).astype(np.uint8),(R//32*32).astype(np.uint8)
    yield 'smooth',cv2.GaussianBlur(L,(0,0),6),cv2.GaussianBlur(R,(0,0),6)
    d=L.copy(); cv2.rectangle(d,(200,80),(500,300),255,-1); cv2.line(d,(0,0),(1240,375),0,3)
    e=R.copy(); cv2.rectangle(e,(180,80),(480,300),255,-1); cv2.line(e,(0,0),(1240,375),0,3)
    yield 'shapes',d,e
cfg=co.make_config(cl,cr)
tot_bad_cv=tot_bad_exact=0; kp_bad=0; n=0
with StereoFrontend(cl,cr) as fe:
    for seed in range(12):
        for name,L,R in variants(seed):
            n+=1
            g=fe.harris_response(L)
            rc=co.harris_response(L)                       # OpenCV operation order
            re=o.harris_response(L,box=o.box7_exact)       # order-independent exact sums
            b1=int((g.view(np.uint32)!=rc.view(np.uint32)).sum()); b2=int((g.view(np.uint32)!=re.view(np.uint32)).sum())
            tot_bad_cv+=b1; tot_bad_exact+=b2
            got=fe.add_new_landmarks(L,R); ref=co.frame(co.stereo_frames(cfg,L,R),0)
            same=len(got['status'])==len(ref['status']) and all(np.array_equal(got[k],ref[k]) for k in ('uv_l','desc_l','status','dist','idx'))
            kp_bad+= (not same)
            if b1 or b2 or not same:
                thr=rc.max()*0.01
                where=np.argwhere(g.view(np.uint32)!=rc.view(np.uint32))
                mx=max(abs(float(g[y,x])) for y,x in where[:2000]) if len(where) else 0
                mx2=max(abs(float(rc[y,x])) for y,x in where[:2000]) if len(where) else 0
                print(seed,name,'GPU!=opencv-order:',b1,'GPU!=exact:',b2,'frame equal:',same,'max |R| at mismatches gpu %.3g cv %.3g thr %.3g'%(mx,mx2,thr))
print('frames',n,'response px GPU!=opencv-order',tot_bad_cv,'GPU!=exact',tot_bad_exact,'frames with different stereo result',kp_bad)
