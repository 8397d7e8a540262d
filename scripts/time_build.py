import os, time, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import raytracingtherestofyourlife_b200 as B
t=time.time(); s=B.Scene.spheres(1000000); print("scene gen", time.time()-t)
ctx=B.Context(0)
t=time.time(); ctx.set_scene(s); ctx.synchronize(); print("set_scene", time.time()-t)
t=time.time(); ctx.build_bvh(); ctx.synchronize(); print("build_bvh", time.time()-t)
