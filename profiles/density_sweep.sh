# grid density (voxels per gridded sphere) x kernel variant on C3 at 8 spp
for d in 2 4 8 16 32; do for v in ${VARIANTS:-0 1}; do echo -n "density $d "; RT_GRID_DENSITY=$d RT_VARIANT=$v python profiles/profile_render.py C3 8 2 2>&1 | grep "launch 1"; done; done
