"""Time axis labels (not on the compute path).

Interface of nemoflux/timeobj.py: TimeObj(nc) finds the variable whose standard_name is 'time' or whose long_name
is 'Time axis' (timeobj.py:8-13); getValues / getSize / getTimeAsDate / getTimeAsString.  The reference gets
calendar objects from xarray; here the raw numbers are decoded from the CF units ('<unit> since Y-M-D').  Mock
data from datagen has no time axis: the reference raises in getTimeAsString (timeobj.py:31-33), this class labels
the step with its index instead.
"""
import datetime
import re

_SECONDS = {'seconds': 1.0, 'minutes': 60.0, 'hours': 3600.0, 'days': 86400.0}
_SINCE = re.compile(r'\s*(seconds|minutes|hours|days)\s+since\s+(\d+)-(\d+)-(\d+)')


_NOLEAP_DAYS = (31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31)


class CalendarDate(object):
    """year / month / day in a CF calendar without a Python equivalent (noleap, 360_day: 30 February exists there)"""

    def __init__(self, year, month, day):
        self.year, self.month, self.day = year, month, day

    def __eq__(self, other):
        return (self.year, self.month, self.day) == (other.year, other.month, other.day)

    def __repr__(self):
        return f'CalendarDate({self.year}, {self.month}, {self.day})'


def _fixed_calendar_date(origin, seconds, calendar):
    """date `seconds` after `origin` in the CF calendars NEMO commonly runs with (xarray decodes them with cftime for
    the reference): noleap / 365_day = no 29 February, 360_day = twelve months of 30 days"""
    days = int((seconds + origin.hour * 3600 + origin.minute * 60 + origin.second) // 86400)
    if calendar == '360_day':
        n = origin.year * 360 + (origin.month - 1) * 30 + (origin.day - 1) + days
        return CalendarDate(n // 360, n % 360 // 30 + 1, n % 30 + 1)
    doy = sum(_NOLEAP_DAYS[:origin.month - 1]) + origin.day - 1 + days
    year, doy = origin.year + doy // 365, doy % 365
    month = 0
    while doy >= _NOLEAP_DAYS[month]:
        doy -= _NOLEAP_DAYS[month]
        month += 1
    return CalendarDate(year, month + 1, doy + 1)


def _is_time_axis(var):
    return getattr(var, 'standard_name', '') == 'time' or getattr(var, 'long_name', '') == 'Time axis'


class TimeObj(object):

    def __init__(self, nc):
        self.timeVarName, self.timeVar, self.units, self.calendar = '', [], '', 'standard'
        self.boundsVar = None
        for name, var in nc.items():
            if _is_time_axis(var):          # the last match wins, as in the reference
                self.timeVarName, self.timeVar, self.units = name, var[:], str(getattr(var, 'units', ''))
                self.calendar = str(getattr(var, 'calendar', 'standard')).lower()
                bnds = str(getattr(var, 'bounds', ''))
                self.boundsVar = nc[bnds][:] if bnds and bnds in nc else None
        since = _SINCE.match(self.units)
        self._origin = datetime.datetime(*(int(since.group(k)) for k in (2, 3, 4))) if since else None
        self._unit_s = _SECONDS[since.group(1)] if since else None

    def getValues(self):
        return self.timeVar[:]

    def getSize(self):
        return len(self.timeVar)

    def getTimeAsDate(self, timeIndex):
        """calendar date of the step, or the index itself when the file has no (decodable) time axis"""
        if self._origin is None or len(self.timeVar) == 0:
            return timeIndex
        seconds = float(self.timeVar[timeIndex]) * self._unit_s
        if self.calendar in ('noleap', '365_day', '360_day'):
            return _fixed_calendar_date(self._origin, seconds, self.calendar)
        return (self._origin + datetime.timedelta(seconds=seconds)).date()

    def getBounds(self):
        """(n, 2) values of the time variable's CF `bounds` variable (NEMO: time_centered_bounds), or None"""
        if self.boundsVar is None or len(self.boundsVar) != len(self.timeVar):
            return None
        return self.boundsVar[:]

    def getTimeAsString(self, timeIndex):
        when = self.getTimeAsDate(timeIndex)
        if isinstance(when, (datetime.date, CalendarDate)):
            return f'{when.year}-{when.month}-{when.day}'
        return f'time index {when}'


def timeWindows(timeObj, nt, spec):
    """window bounds [b0 = 0 < b1 < ... < bK = nt] of the nt steps for time means (fluxSection(windows=)):
    spec an int N -> windows of N steps (the last one holds what is left); 'month' / 'year' -> runs of consecutive
    steps with the same (year, month) / year of getTimeAsDate, in every calendar it decodes (standard, noleap /
    365_day, 360_day).  Calendar windows need a time axis of nt values with CF units '<unit> since Y-M-D'."""
    if isinstance(spec, str) and spec.strip().isdigit():
        spec = int(spec)
    if isinstance(spec, int) and not isinstance(spec, bool):
        if spec < 1:
            raise ValueError(f'a time window holds at least 1 step, got {spec}')
        return list(range(0, nt, spec)) + [nt] if nt > 0 else [0]
    if spec not in ('month', 'year'):
        raise ValueError(f"time windows: expected a number of steps, 'month' or 'year', got {spec!r}")
    if timeObj is None or timeObj._origin is None or timeObj.getSize() != nt or nt == 0:
        raise ValueError(f"time windows by {spec} need a time axis of {nt} steps with CF units '<unit> since Y-M-D' "
                         "(this file has none): give a number of steps instead")
    dates = [timeObj.getTimeAsDate(i) for i in range(nt)]
    keys = [(d.year, d.month) if spec == 'month' else d.year for d in dates]
    return [0] + [i for i in range(1, nt) if keys[i] != keys[i - 1]] + [nt]
