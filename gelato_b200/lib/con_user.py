"""/root/reference/lib/con_user.py:33-42 -- user constraints.  Registered built-ins run on the GPU
(gelato_b200.lib.configure(user_eq=OrbitAtEvent("IIP_END", [("perigee_radius", 6378137.0, 1.0)]), ...): orbit
quantities of the state at a named event, one to three rows, see plan.OrbitAtEvent / ORBIT_QUANTITIES; result-table
columns at a named event, plan.TableAtEvent / TABLE_COLUMNS; or a list of them); without one
the group is absent (None), like a user_constraints.py that returns None.  An arbitrary Python callable stays on the
host: lib/jac_fd.py runs the reference's loop over it."""
from . import _jacobian, _value

equality_user = _value("eqcon_user")
inequality_user = _value("ineqcon_user")
equality_jac_user = _jacobian("eqcon_user")  # :33
inequality_jac_user = _jacobian("ineqcon_user")  # :39
