import os, sys, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests import oracle_lib as O, ref_lib as R
rng=np.random.default_rng(301)
for lg in (1,2):
    msg=O.rand_field(rng,(1,1<<lg))
    ref,_=R.batch_coset_dft(msg,2)
    exp=O.rs_encode(msg,2)
    print("lg",lg,"msg",O.from_monty(msg),"\n ref",O.from_monty(ref),"\n exp",O.from_monty(exp))
